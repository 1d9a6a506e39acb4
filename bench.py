#!/usr/bin/env python
"""bench.py -- GE2E train steps/sec (and d-vectors/sec) on N B200s, one process per GPU.

    python bench.py [--gpus N] [--steps K] [--warmup W]            # this framework (CUDA, sm_100a)
    python bench.py --impl reference [--steps K] [--warmup W]       # the unmodified reference on the host cores
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W      # N > 1

Workload (BASELINE.json configs[1]): one GE2E training step = encoder forward + GE2E loss + backward
+ gradient clip 1.0 + RAdam (lr 2e-3, eps 1e-6) with Modified-Noam(4000), on a synthetic batch of
64 speakers x 15 utterances x T frames x 80 mel bins, one T drawn from [140, 180] per step
(Datasets.py:77-84), dropout on (train mode).  N > 1: every rank owns its own 64 speakers (rank-local
loss, SURVEY.md D8) and the flat gradient arena is averaged with one NCCL all-reduce -> weak scaling.

One JSON line is printed by rank 0.  `value` is measured with inputs resident in HBM; `e2e` includes
the pinned-host -> device copy of every batch and a device -> host read of the loss every step.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SPEAKERS, UTTS, MEL = 64, 15, 80
T_MIN, T_MAX = 140, 180


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(hbm=p["hbm_gbs"], tf_burst=p["bf16_tflops"], tf_sus=p["bf16_tflops_sustained"], src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sus=1400.0, src="fallback")


def synth_mel(gen, batch, frames, device):
    """Log-mel-like features: clamp(-5 + 2 randn, ln 1e-5, 2)  (SURVEY.md 8d)."""
    x = torch.randn(batch, MEL, frames, generator=gen, device=device) * 2.0 - 5.0
    return x.clamp_(float(np.log(1e-5)), 2.0)


def dense_flops_fwd(T):
    """Algorithmic forward FLOPs per slice as the reference executes it (SURVEY.md 8d, dense accounting)."""
    return 40960.0 * T + 3 * (1572864.0 * T + 1024.0 * T * T) + 131072.0


def min_flops_fwd(T):
    """Forward FLOPs per slice of the variant executed here: last layer pruned to the t = 0 query (SURVEY.md 8d F_min)."""
    return 40960.0 * T + 2 * (1572864.0 * T + 1024.0 * T * T) + (262144.0 * T + 1024.0 * T + 1310720.0) + 131072.0


class ClockSampler:
    """SM clock and throttle reasons DURING the timed region: an NVML polling thread (5 ms period; the timed region of a
    default run is only ~130 ms, too short for `nvidia-smi -lms`), falling back to nvidia-smi when NVML is missing."""

    REASONS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20),
               ("sw_power_cap", 0x4))

    def __init__(self, index):
        self.index, self.rows, self.proc, self.thread = index, [], None, None
        self.stop = threading.Event()
        self.nvml = None
        self.err = None

    def _handle(self):
        import pynvml
        pynvml.nvmlInit()
        try:
            pr = torch.cuda.get_device_properties(self.index)
            bus = "%08x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
            h = pynvml.nvmlDeviceGetHandleByPciBusId(bus.encode())
        except Exception:
            h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
        return pynvml, h

    def sample(self):
        """One NVML reading now (also called from the main thread while the GPU is still busy with the timed steps, so a
        starved polling thread cannot leave the line without clocks)."""
        if self.nvml is None:
            return
        pynvml, h = self.nvml, self.h
        try:
            if self.mx is None:
                self.mx = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
            sm = pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
            try:
                mask = pynvml.nvmlDeviceGetCurrentClocksEventReasons(h)
            except Exception:
                mask = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
            self.rows.append((float(sm), float(self.mx) if self.mx else None, int(mask)))
        except Exception as ex:      # keep polling; the summary reports the last error if nothing was sampled
            self.err = repr(ex)

    def _poll(self):
        while not self.stop.is_set():
            self.sample()
            self.stop.wait(0.005)

    def __enter__(self):
        try:
            pynvml, h = self._handle()
            self.nvml, self.h, self.mx = pynvml, h, None
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return self
        except Exception as ex:
            self.nvml = None
            self.err = repr(ex)
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            c = [x.strip() for x in line.split(",")]
            try:
                mask = 0
                for (n, bit), v in zip(self.REASONS, c[3:7]):
                    if v.lower().startswith("active"):
                        mask |= bit
                self.rows.append((float(c[0]), float(c[1]), mask))
            except (ValueError, IndexError):
                continue

    def __exit__(self, *a):
        if self.nvml is not None:
            self.stop.set()
            self.thread.join(timeout=2)
        elif self.proc is not None:
            time.sleep(0.25)
            self.proc.terminate()
            self.thread.join(timeout=2)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0, "error": self.err}
        sm = [r[0] for r in self.rows]
        mx = [r[1] for r in self.rows if r[1]]
        mask = 0
        for r in self.rows:
            mask |= r[2]
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(n for n, bit in self.REASONS if mask & bit), "samples": len(sm),
                "source": "nvml" if self.nvml is not None else "nvidia-smi"}


# ------------------------------------------------------------------------------------------------
# reference arm / CPU baseline: the UNMODIFIED reference (baseline/_ref, staged by __graft_entry__.build()) on the
# host cores -- its `Device: '-1'` path (Train.py:34-35, README.md:56-58).  Falls back to the oracle port when the
# staged copy is missing.

REF_COPY = os.path.join(ROOT, "baseline", "_ref")


def step_lengths(count):
    """One frame count per step (Datasets.py:77-84), the same sequence for every arm and every rank."""
    rs = np.random.RandomState(0)
    return [int(rs.randint(T_MIN, T_MAX + 1)) for _ in range(count)]


class ReferenceTrainer:
    """Trainer.Train_Step (Train.py:140-168) with the published optimiser pair (RAdam + Modified_Noam_Scheduler,
    SURVEY.md D4) driving the reference's own GE2E / GE2E_Loss / RAdam / scheduler classes, unmodified, on CPU."""

    def __init__(self):
        import yaml
        if REF_COPY not in sys.path:
            sys.path.insert(0, REF_COPY)
        import warnings
        warnings.filterwarnings("ignore")
        from Modules import GE2E, GE2E_Loss                      # baseline/_ref/Modules.py
        from Radam import RAdam                                  # baseline/_ref/Radam.py
        from Noam_Scheduler import Modified_Noam_Scheduler       # baseline/_ref/Noam_Scheduler.py
        from Arg_Parser import Recursive_Parse
        import Modules
        assert os.path.dirname(os.path.abspath(Modules.__file__)) == REF_COPY, Modules.__file__
        hp = Recursive_Parse(yaml.load(open(os.path.join(REF_COPY, "Hyper_Parameters.yaml")), Loader=yaml.Loader))
        self.cores = os.cpu_count() or 1
        torch.set_num_threads(self.cores)
        torch.manual_seed(0)
        self.model = GE2E(hp).train()
        self.criterion = GE2E_Loss()
        self.optimizer = RAdam(self.model.parameters(), lr=2e-3, betas=(0.9, 0.999), eps=1e-6, weight_decay=0.0)
        self.scheduler = Modified_Noam_Scheduler(self.optimizer, base=4000)
        self.gen = torch.Generator().manual_seed(1234)

    def step(self, speakers, frames):
        features = synth_mel(self.gen, speakers * UTTS, frames, "cpu")
        embeddings = self.model(features)
        loss = self.criterion(embeddings, UTTS)
        self.optimizer.zero_grad()
        loss.backward()
        torch.nn.utils.clip_grad_norm_(parameters=self.model.parameters(), max_norm=1.0)
        self.optimizer.step()
        self.scheduler.step()
        return loss.item()


def reference_train_step_rate(steps, warmup, lengths):
    """steps/s of the full 64 x 15 batch on the host cores; every step is timed on the whole batch."""
    tr = ReferenceTrainer()
    tr.step(2, 32)                                     # thread pool / allocator warm-up, not a benchmark step
    for i in range(warmup):
        tr.step(SPEAKERS, lengths[i])
    t0 = time.perf_counter()
    for i in range(steps):
        tr.step(SPEAKERS, lengths[warmup + i])
    dt = (time.perf_counter() - t0) / steps
    sample = "full batch: 64 speakers x 15 utt x T~U[140,180] per step, %d timed step(s), dropout on" % steps
    return 1.0 / dt, dt * 1e3, tr.cores, sample, "reference"


def port_train_step_rate(steps, warmup, lengths):
    """Fallback when baseline/_ref is absent: the oracle's restatement of the same step."""
    from oracle import ge2e_oracle as O
    from oracle import synth
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    state = O.to_torch_state(synth.make_state(0), torch.float32, requires_grad=True)
    params = [v for k, v in state.items() if v.requires_grad]
    w = torch.tensor(10.0, requires_grad=True)
    b = torch.tensor(-5.0, requires_grad=True)
    gen = torch.Generator().manual_seed(1234)
    m = [torch.zeros_like(p) for p in params]
    v = [torch.zeros_like(p) for p in params]

    def one_step(spk, frames, step):
        mel = torch.as_tensor(synth.make_mel(step, spk * UTTS, frames))
        for p in params:
            p.grad = None
        d = O.encoder_forward(state, mel, 1, dropout_p=0.1, gen=gen)
        loss = O.ge2e_loss(d, UTTS, w, b)
        loss.backward()
        total = torch.sqrt(sum((p.grad.double() ** 2).sum() for p in params)).item()
        coef = O.clip_coef(total, 1.0)
        lr = O.modified_noam_lr(2e-3, step, 4000)
        with torch.no_grad():
            for p, mi, vi in zip(params, m, v):
                O.radam_step(p.detach().numpy(), (p.grad * coef).numpy(), mi.numpy(), vi.numpy(), step + 1, lr,
                             eps=1e-6)
        return float(loss.detach())

    one_step(2, 32, 0)
    for i in range(warmup):
        one_step(SPEAKERS, lengths[i], i)
    t0 = time.perf_counter()
    for i in range(steps):
        one_step(SPEAKERS, lengths[warmup + i], warmup + i)
    dt = (time.perf_counter() - t0) / steps
    sample = "full batch: 64 speakers x 15 utt x T~U[140,180] per step, %d timed step(s), dropout on" % steps
    return 1.0 / dt, dt * 1e3, cores, sample, "port"


def cpu_train_step_rate(steps, warmup, lengths):
    if os.path.exists(os.path.join(REF_COPY, "Modules.py")):
        return reference_train_step_rate(steps, warmup, lengths)
    return port_train_step_rate(steps, warmup, lengths)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps, warmup = max(1, args.steps), max(0, args.warmup)
    lengths = step_lengths(max(3, warmup) + steps)[max(3, warmup) - warmup:]     # the native arm's timed lengths
    rate, ms, cores, sample, kind = cpu_train_step_rate(steps, warmup, lengths)
    line = {
        "impl": "reference", "metric": "GE2E train steps/sec (64 spk x 15 utt, fwd+bwd+clip+RAdam/Noam)",
        "value": rate, "unit": "steps/s", "n_gpus": args.gpus, "steps": steps, "warmup": warmup,
        "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": "ge2e_train_step_64x15_T140-180", "speakers_per_gpu": SPEAKERS,
                   "utterances_per_speaker": UTTS, "frames": "one T~U[140,180] per step", "mel": MEL,
                   "optimizer": "reference RAdam lr2e-3 eps1e-6 + Modified_Noam(4000), clip 1.0", "dropout": 0.1,
                   "device": "cpu (reference Device -1 path), %d threads" % cores},
        "cpu_baseline": {"value": rate, "unit": "steps/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": rate, "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def dump_outputs(out_dir, arrays):
    """Write every tensor of ``arrays`` as ``out_dir/<name>.npy`` in float32."""
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy())


# ------------------------------------------------------------------------------------------------
def run_native(args):
    import torch.distributed as dist
    from speaker_embedding_torch_b200 import GE2E, GE2E_Loss, _native
    from speaker_embedding_torch_b200.Arg_Parser import default_hyper_parameters
    from speaker_embedding_torch_b200.Noam_Scheduler import Modified_Noam_Scheduler
    from speaker_embedding_torch_b200.Radam import RAdam
    from speaker_embedding_torch_b200.distributed import apply_gradient_allreduce

    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device (B200); there is no CPU path. "
                           "Use --impl reference for the CPU baseline.")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import datetime
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=240))
    K, W = max(1, args.steps), max(3, args.warmup)
    pk = peaks()

    torch.manual_seed(0)
    model = GE2E(default_hyper_parameters())
    with torch.no_grad():                      # perturb every tensor so no layer / bias is degenerate (SURVEY D11)
        g0 = torch.Generator().manual_seed(1)
        for p in model.parameters():
            p.add_(0.1 * torch.randn(p.shape, generator=g0) * (p.abs().mean() + 0.05))
    model = model.to(dev).train()
    crit = GE2E_Loss().to(dev)
    if world > 1:
        apply_gradient_allreduce(model)
    opt = RAdam(model.parameters(), lr=2e-3, betas=(0.9, 0.999), eps=1e-6, weight_decay=0.0, max_grad_norm=1.0)
    sched = Modified_Noam_Scheduler(opt, base=4000)

    lengths = step_lengths(W + K + 4)
    # the warm-up covers the longest and the shortest slice, so that every kernel instantiation (CUDA loads kernels
    # lazily) and the largest workspace exist before the timed region, as they do after the first minutes of training
    lengths[0], lengths[1] = T_MAX, T_MIN
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    batch = SPEAKERS * UTTS

    last = {}

    def step(mel):
        opt.zero_grad(set_to_none=True)
        d = model(mel)
        loss = crit(d, UTTS)
        loss.backward()
        opt.step()
        sched.step()
        last["dvectors"] = d
        return loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident inputs: `value`
    dev_mels = [synth_mel(gen, batch, T, dev) for T in lengths[:W + K]]
    for i in range(W):
        step(dev_mels[i])
    for i in range(5):                      # a few more untimed steps: clocks / allocator / NCCL reach steady state
        step(dev_mels[i % W])
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local) as clk:
        e0.record()
        for i in range(K):
            loss = step(dev_mels[W + i])
        e1.record()
        clk.sample()                        # the queue is still draining: a reading inside the timed region
        barrier()
    ms = e0.elapsed_time(e1)
    t = torch.tensor([ms], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    value = world * K / (ms_total * 1e-3)
    last_loss = float(loss.item())
    if args.dump_outputs and rank == 0:
        arrays = {"loss": loss.reshape(1), "dvectors": last["dvectors"]}
        for n, p in model.named_parameters():
            arrays["param." + n] = p
            arrays["grad." + n] = p.grad
        dump_outputs(args.dump_outputs, arrays)
    del dev_mels

    # ---- end to end through the public API: pinned host batch -> H2D -> step -> loss D2H
    # (the same frame counts as the device-resident pass, so that `e2e` and `value` time the same work)
    host = [synth_mel(gen, batch, T, dev).cpu().pin_memory() for T in lengths[W:W + K]]
    from speaker_embedding_torch_b200.Prefetch import Device_Prefetcher
    feeder = Device_Prefetcher(host, dev, reserve_bytes=batch * 80 * T_MAX * 4)     # buffers sized for Frame_Length.Max
    # the loss of every step is copied to pinned host memory inside the timed region (non-blocking, like the reference's
    # `scalar_Dict['Train']['Loss'] += loss`, Train.py:163, which does not stall the loop); the host reads them afterwards
    loss_host = torch.zeros(K, dtype=torch.float32).pin_memory()
    barrier()
    e0.record()
    for i, mel in enumerate(feeder):             # batch i+1 crosses PCIe on a side stream while batch i is computed
        loss_host[i:i + 1].copy_(step(mel).detach().reshape(1), non_blocking=True)
    e1.record()
    barrier()
    lv = float(loss_host.sum().item())
    assert lv == lv, "NaN loss in the end-to-end pass"
    t = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = world * K / (float(t.item()) * 1e-3)
    h2d = int(np.mean([h.numel() * 4 for h in host]))
    del host

    # ---- per-kernel profile (events around every launch; separate pass so it does not perturb `value`), at a FIXED
    # frame count (160, the centre of the range) so that the committed ncu DRAM-traffic capture describes the same launch
    line_extra = {}
    # every rank runs the profiled steps (backward contains the gradient all-reduce); rank 0 reports
    prof_steps, Tprof = 2, 160
    mel_prof = synth_mel(gen, batch, Tprof, dev)
    step(mel_prof)                               # allocator / lazy-load warm-up at this frame count
    torch.cuda.synchronize()
    _native.prof_enable(True)
    for i in range(prof_steps):
        step(mel_prof)
    torch.cuda.synchronize()
    rep = _native.prof_report()
    _native.prof_enable(False)
    del mel_prof
    barrier()

    def is_contraction(tag):
        return tag.startswith("gemm.") or tag.startswith("attn_fused") or tag.startswith("attn_train")

    if rank == 0:
        launches_per_step = sum(r["launches"] for r in rep.values()) // prof_steps
        tot_ms = sum(r["ms"] for r in rep.values())
        tag, r = max(rep.items(), key=lambda kv: kv[1]["ms"])
        per_launch_ms = r["ms"] / r["launches"]
        tflops = r["flops"] / r["launches"] / (per_launch_ms * 1e-3) / 1e12
        gbs = r["bytes"] / r["launches"] / (per_launch_ms * 1e-3) / 1e9
        # SURVEY.md 8(d): every dense contraction of the encoder is charged against the sustained bf16 tensor peak with its
        # 16-bit dense FLOP count (the extra MMAs of the split-plane products are not credited); row kernels against HBM
        tensor_bound = is_contraction(tag) and r["flops"] > 0
        roof = {"kernel": tag, "bound": "tensor" if tensor_bound else "hbm",
                "achieved": tflops if tensor_bound else gbs, "peak": pk["tf_sus"] if tensor_bound else pk["hbm"],
                "unit": "TFLOP/s" if tensor_bound else "GB/s", "traffic": None,
                "peak_source": pk["src"] + (" sustained bf16" if tensor_bound else " copy"),
                "launch_ms": per_launch_ms, "share_of_step": r["ms"] / tot_ms, "frames": Tprof,
                "alg_flops_per_launch": r["flops"] / r["launches"], "alg_bytes_per_launch": r["bytes"] / r["launches"]}
        try:      # DRAM bytes per launch of the same kernel at the same frame count, from the committed ncu capture
            tr = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))
            if tr.get("frames") == Tprof and tag in tr:
                roof["traffic"] = tr[tag]["read"] + tr[tag]["write"]
                roof["traffic_source"] = tr.get("source", "profiles/r02_traffic.json")
        except (OSError, ValueError, KeyError):
            pass
        roof["frac"] = roof["achieved"] / roof["peak"]
        # the whole step against the same peak: F_min FLOPs of forward + backward (3 x forward) at the mean frame count of
        # the timed steps / measured step time
        mean_fl = float(np.mean([min_flops_fwd(T) for T in lengths[W:W + K]]))
        step_tf = 3 * batch * mean_fl * (value / world) / 1e12
        roof["step"] = {"achieved": step_tf, "peak": pk["tf_sus"], "unit": "TFLOP/s", "frac": step_tf / pk["tf_sus"],
                        "alg_flops_per_step": 3 * batch * mean_fl,
                        "accounting": "3 x F_min(T) x 960 slices, SURVEY.md 8(d); extra split-plane MMAs not credited"}
        breakdown = {k: {"ms_per_step": round(v["ms"] / prof_steps, 4), "launches": v["launches"] // prof_steps,
                         "tflops": round(v["flops"] / (v["ms"] * 1e-3) / 1e12, 2) if v["flops"] else 0.0,
                         "gbs": round(v["bytes"] / (v["ms"] * 1e-3) / 1e9, 1)}
                     for k, v in sorted(rep.items(), key=lambda kv: -kv[1]["ms"])}
        line_extra = {"roofline": roof, "gpu_launches": launches_per_step * K, "breakdown": breakdown,
                      "profiled_step_ms": tot_ms / prof_steps, "profiled_T": Tprof}

    # ---- inference metrics of BASELINE.json on every rank (utterance shards, no collective; max over ranks):
    #      d-vectors/s on 160-frame slices and config 3 (5 x 64-frame slices, 32 overlap) incl. its end-to-end path
    infer = run_infer_shard(model, gen, dev, world, rank, barrier, dist)
    if rank == 0:
        dv_ms = infer.pop("_dv_ms")
        _native.prof_enable(True)
        model.eval()
        with torch.no_grad():
            model(synth_mel(gen, batch, 160, dev))
        torch.cuda.synchronize()
        irep = _native.prof_report()
        _native.prof_enable(False)
        model.train()
        line_extra["infer"] = infer
        line_extra["infer_breakdown"] = {k: {"ms": round(v["ms"], 4), "launches": v["launches"],
                                             "tflops": round(v["flops"] / (v["ms"] * 1e-3) / 1e12, 2) if v["flops"] else 0.0,
                                             "gbs": round(v["bytes"] / (v["ms"] * 1e-3) / 1e9, 1)}
                                         for k, v in sorted(irep.items(), key=lambda kv: -kv[1]["ms"])}
        line_extra["extra"] = {"flop_accounting": "F_min (last layer pruned to the t=0 query), 16-bit dense count, extra split-plane MMAs not credited",
                               "infer_tensor_frac_of_sustained": batch * min_flops_fwd(160) / (dv_ms * 1e-3) / 1e12 / pk["tf_sus"],
                               "train_precision": int(model.train_precision), "last_loss": last_loss}

    barrier()
    if rank == 0:
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            try:   # bounded sample: two full-batch steps of the reference on the host cores (~15-20 s)
                rate, cms, cores, sample, kind = cpu_train_step_rate(2, 0, lengths[W:W + 2])
                cpu = {"value": rate, "unit": "steps/s", "cores": cores, "kind": kind, "sample": sample}
            except Exception as exc:  # the baseline must never take the GPU number down with it
                cpu = {"value": None, "unit": "steps/s", "cores": os.cpu_count(), "kind": "reference",
                       "sample": "failed: %r" % (exc,)}
        line = {
            "metric": "GE2E train steps/sec (64 spk x 15 utt, fwd+bwd+clip+RAdam/Noam)",
            "value": value, "unit": "steps/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f16 (operands split into %d fp16 planes forward / 2 backward = fp32-class mantissa, fp32 accumulate)" % int(model.train_precision),
            "data": "synthetic",
            "config": {"workload": "ge2e_train_step_64x15_T140-180", "speakers_per_gpu": SPEAKERS,
                       "utterances_per_speaker": UTTS, "frames": "one T~U[140,180] per step", "mel": MEL,
                       "optimizer": "fused RAdam lr2e-3 eps1e-6 + Modified_Noam(4000), clip 1.0",
                       "dropout": 0.1, "parallelism": "dp%d" % world,
                       "l2": "per-step working set (>5 GB of activations) exceeds the 126 MB L2; no flush needed"},
            "clocks": clk.summary(),
            "e2e": {"value": e2e_value, "unit": "steps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                    "readback": "the loss of every step -> pinned host memory, non-blocking, inside the timed region"},
            "cpu_baseline": cpu,
        }
        line.update(line_extra)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def run_infer_shard(model, gen, dev, world, rank, barrier, dist, utt=4000, reps=25):
    """BASELINE config 3 on this rank's shard: `utt` utterances per step, 5 x 64-frame slices at 32 overlap
    (Inference.py:95-115), `reps` timed steps (25 x 4 000 = the 100 000 utterances of the configuration, per GPU); plus the 160-frame single-slice d-vector rate.  Returns rank-0 dict
    with whole-job numbers (time = max over ranks; utterances are independent, there is no collective)."""
    from speaker_embedding_torch_b200.Prefetch import Device_Prefetcher
    pk = peaks()
    batch = SPEAKERS * UTTS
    S, F, O = 5, 64, 32
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def max_ms(ms):
        t = torch.tensor([ms], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    model.eval()
    with torch.no_grad():
        mel160 = synth_mel(gen, batch, 160, dev)
        for _ in range(3):
            model(mel160)
        barrier()
        e0.record()
        for _ in range(10):
            model(mel160)
        e1.record()
        barrier()
        dv_ms = max_ms(e0.elapsed_time(e1)) / 10
        del mel160
        windows = synth_mel(gen, utt, S * (F - O) + O, dev)                      # [utt, 80, 192]
        for _ in range(3):
            model.embed_windows(windows, F, O)
        barrier()
        e0.record()
        for _ in range(reps):
            out = model.embed_windows(windows, F, O)
        e1.record()
        barrier()
        ms = max_ms(e0.elapsed_time(e1))
        # end to end: fp16 192-frame windows (as the reference stores its patterns, Pattern_Generator.py:123) cross PCIe
        # through Device_Prefetcher, slices are cut and upcast inside the prenet load, d-vectors are read back
        host_windows = windows.half().cpu().pin_memory()
        feeder = Device_Prefetcher([host_windows] * reps, dev, reserve_bytes=host_windows.numel() * 2)
        host_out = [torch.empty(utt, 256).pin_memory() for _ in range(reps)]
        model.embed_windows(windows.half(), F, O)
        barrier()
        e0.record()
        for i, w in enumerate(feeder):
            host_out[i].copy_(model.embed_windows(w, F, O), non_blocking=True)
        e1.record()
        barrier()
        ms_e2e = max_ms(e0.elapsed_time(e1))
        checksum = float(out.float().sum().item())
    model.train()
    if rank != 0:
        return {}
    flops = utt * S * min_flops_fwd(F)
    return {"_dv_ms": dv_ms,
            "dvectors_per_sec_160f": world * batch / (dv_ms * 1e-3), "ms_per_960x160_batch": dv_ms,
            "config3": {"metric": "utterances/sec, multi-slice extraction 5 x 64 frames / 32 overlap",
                        "value": world * reps * utt / (ms * 1e-3), "unit": "utterances/s",
                        "utterances_per_step_per_gpu": utt, "utterances_per_gpu": utt * reps, "steps": reps, "ms_per_step": ms / reps, "n_gpus": world,
                        "sharding": "utterance shards, no collective",
                        "e2e": {"value": world * reps * utt / (ms_e2e * 1e-3), "unit": "utterances/s",
                                "h2d_bytes_per_step": host_windows.numel() * 2, "d2h_bytes_per_step": utt * 256 * 4},
                        "tensor_frac_of_sustained": flops * reps / (ms * 1e-3) / 1e12 / pk["tf_sus"],
                        "dvec_checksum": checksum}}


def run_infer(args):
    """Config 3: batched multi-slice extraction (5 x 64-frame slices, 32 overlap => 192-frame windows per
    utterance, Inference.py:95-115).  Utterances are independent: rank r embeds its own shard, no collective.
    A step = one chunk of 4000 utterances per GPU; value = utterances/s over all ranks."""
    import torch.distributed as dist
    from speaker_embedding_torch_b200 import GE2E
    from speaker_embedding_torch_b200.Arg_Parser import default_hyper_parameters
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import datetime
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=240))
    K, W = max(1, args.steps), max(3, args.warmup)
    torch.manual_seed(0)
    model = GE2E(default_hyper_parameters()).to(dev).eval()
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    utt, S, F, O = 4000, 5, 64, 32
    windows = synth_mel(gen, utt, S * (F - O) + O, dev)                      # [utt, 80, 192]
    # the collater's overlapping slices (stride F - O), utterance-major rows
    chunk = torch.stack([windows[:, :, i * (F - O):i * (F - O) + F] for i in range(S)], dim=1).reshape(utt * S, MEL, F).contiguous()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    with torch.no_grad():
        for _ in range(W):
            model(chunk, S)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with ClockSampler(local) as clk:
            e0.record()
            for _ in range(K):
                out = model(chunk, S)
            e1.record()
            clk.sample()
            barrier()
        t = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        # end to end: the un-sliced 192-frame windows cross PCIe (pinned host -> Device_Prefetcher, next chunk in flight
        # while this one is embedded), the collater's overlapping slices are cut on the device, d-vectors come back
        from speaker_embedding_torch_b200.Modules import Overlapped_Slices
        from speaker_embedding_torch_b200.Prefetch import Device_Prefetcher
        # patterns travel as the reference stores them (fp16, Pattern_Generator.py:123); slicing and the upcast happen
        # inside the prenet's input load (GE2E.embed_windows -> spk_encoder_forward_view)
        host_windows = windows.half().cpu().pin_memory()
        assert torch.equal(Overlapped_Slices(windows, F, O), chunk)
        feeder = Device_Prefetcher([host_windows] * K, dev, reserve_bytes=host_windows.numel() * 2)
        host_out = [torch.empty(utt, 256).pin_memory() for _ in range(K)]       # d-vectors land here, no per-step sync
        model.embed_windows(windows.half(), F, O)                               # warm-up of the fp16 load
        barrier()
        e0.record()
        for i, w in enumerate(feeder):
            host_out[i].copy_(model.embed_windows(w, F, O), non_blocking=True)
        e1.record()
        barrier()
        assert abs(float(host_out[-1].sum()) - float(out.float().sum().item())) < 2e-2 * utt   # fp16 patterns
        t2 = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(t2, op=dist.ReduceOp.MAX)
    if rank == 0:
        pk = peaks()
        flops = utt * S * min_flops_fwd(F)
        print(json.dumps({
            "metric": "utterances/sec, multi-slice d-vector extraction (5 x 64 frames, 32 overlap)",
            "value": world * K * utt / (ms * 1e-3), "unit": "utterances/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f16 operands, fp32 accumulate", "data": "synthetic",
            "config": {"workload": "multislice_inference_5x64_o32", "utterances_per_step_per_gpu": utt,
                       "parallelism": "dp%d (utterance shards, no collective)" % world},
            "clocks": clk.summary(),
            "e2e": {"value": world * K * utt / (float(t2.item()) * 1e-3), "unit": "utterances/s",
                    "h2d_bytes_per_step": host_windows.numel() * 2, "d2h_bytes_per_step": utt * 256 * 4},
            "extra": {"tensor_frac_of_sustained": flops * K / (ms * 1e-3) / 1e12 / pk["tf_sus"],
                      "dvec_checksum": float(out.float().sum().item())},
        }))
    if world > 1:
        dist.destroy_process_group()


def _ge2e_graph_us(emb, crit, N, M, D, reps):
    """Device time of one spk_ge2e_loss call (forward + backward in one call): `reps` calls through the C ABI captured in
    a CUDA graph, the replay timed with CUDA events on the replay stream.  The per-stage event sums of the library's
    profiler put an event pair around every launch, which costs more than the small launches themselves; this is the
    figure a training step sees (the loss runs between the head kernels and the encoder backward on one stream, with
    its input still in L2).  None when the capture fails."""
    import ctypes
    from speaker_embedding_torch_b200 import _native as NV
    try:
        lib = NV.lib()
        wsb = lib.spk_ge2e_workspace_bytes(N, M)
        ws = torch.empty(wsb, dtype=torch.uint8, device="cuda")
        scal = torch.zeros(3, dtype=torch.float32, device="cuda")
        d_emb = torch.empty_like(emb)
        wt, bs = crit.weight.detach().float().contiguous(), crit.bias.detach().float().contiguous()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())

        def call():
            NV.check(lib.spk_ge2e_loss(NV.ptr(emb), N, M, D, NV.ptr(wt), NV.ptr(bs), ctypes.c_void_p(scal.data_ptr()),
                                       NV.ptr(d_emb), ctypes.c_void_p(scal.data_ptr() + 4),
                                       ctypes.c_void_p(scal.data_ptr() + 8), NV.ptr(ws), wsb,
                                       NV.stream_ptr(emb.device)), "spk_ge2e_loss")
        with torch.cuda.stream(side):
            for _ in range(3):
                call()
            side.synchronize()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph, stream=side):
                for _ in range(reps):
                    call()
            graph.replay()
            side.synchronize()
            best = None
            for _ in range(3):
                t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                t0.record(side)
                graph.replay()
                t1.record(side)
                side.synchronize()
                dt = t0.elapsed_time(t1) * 1e3 / reps
                best = dt if best is None else min(best, dt)
        torch.cuda.current_stream().wait_stream(side)
        return best
    except Exception as exc:                                   # noqa: BLE001 -- report, fall back to the stage events
        print("ge2e graph timing unavailable for N=%d: %s" % (N, exc), file=sys.stderr)
        try:
            torch.cuda.synchronize()
        except Exception:                                      # noqa: BLE001
            pass
        return None


def run_ge2e(args):
    """BASELINE config 5: fused GE2E loss forward + backward, N = 64 .. 4096 speakers x 15 utterances x 256-d.
    One JSON line: per N the device time of the library's launches (CUDA events around every kernel), the algorithmic
    bytes (2 N M D 4: read E, write dE) and FLOPs (6 N M N D), the binding roofline side and the fraction reached."""
    from speaker_embedding_torch_b200 import GE2E_Loss, _native
    if int(os.environ.get("RANK", "0")) != 0:
        return
    torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
    pk = peaks()
    crit = GE2E_Loss().cuda()
    M, D = 15, 256
    rows = []
    for N in (64, 128, 256, 512, 1024, 2048, 4096):
        torch.manual_seed(N)
        e = torch.nn.functional.normalize(torch.randn(N * M, D, device="cuda"), dim=1).requires_grad_(True)
        for _ in range(max(3, args.warmup)):
            e.grad = None
            crit(e, M).backward()
        torch.cuda.synchronize()
        iters = max(5, args.steps) if N <= 1024 else 5
        _native.prof_enable(True)
        for _ in range(iters):
            e.grad = None
            loss = crit(e, M)
            loss.backward()
        torch.cuda.synchronize()
        rep = _native.prof_report()
        _native.prof_enable(False)
        us_stages = sum(v["ms"] for k, v in rep.items() if k.startswith("ge2e")) / iters * 1e3
        launches = sum(v["launches"] for k, v in rep.items() if k.startswith("ge2e")) // iters
        if N < 256:
            launches = 3          # one profiler scope around the three stage kernels of the small-N path
        us_graph = _ge2e_graph_us(e.detach(), crit, N, M, D, reps=20 if N <= 1024 else 4)
        us = us_graph if us_graph is not None else us_stages
        us_no_pdl = None
        if N < 256 and us_graph is not None:                   # A/B of the programmatic dependent launch of stages 2, 3
            _native.set_option("ge2e_dependent_launch", 0)
            try:
                us_no_pdl = _ge2e_graph_us(e.detach(), crit, N, M, D, reps=20)
            finally:
                _native.set_option("ge2e_dependent_launch", 1)
        nbytes, flops = 2.0 * N * M * D * 4, 6.0 * N * M * N * D
        t_hbm, t_tc = nbytes / (pk["hbm"] * 1e9), flops / (pk["tf_burst"] * 1e12)
        bound = "hbm" if t_hbm > t_tc else "tensor"
        achieved = nbytes / us / 1e3 if bound == "hbm" else flops / us / 1e6
        peak = pk["hbm"] if bound == "hbm" else pk["tf_burst"]
        rows.append({"N": N, "M": M, "us": round(us, 1), "us_sum_of_stage_events": round(us_stages, 1),
                     "timing": "graph replay" if us_graph is not None else "stage events",
                     "us_without_dependent_launch": None if us_no_pdl is None else round(us_no_pdl, 1),
                     "stage_events_us": {k: round(v["ms"] / iters * 1e3, 1) for k, v in sorted(rep.items())
                                         if k.startswith("ge2e")},
                     "launches": launches, "loss": round(loss.item(), 5),
                     "alg_GBps": round(nbytes / us / 1e3, 1), "alg_TFLOPs": round(flops / us / 1e6, 2),
                     "roofline_us": round(max(t_hbm, t_tc) * 1e6, 2), "bound": bound,
                     "frac": round(achieved / peak, 4),
                     "path": "fused SIMT kernel (3 stream-ordered stages, 8-row tiles)" if N < 256 else "tcgen05 GEMM composition"})
    print(json.dumps({"metric": "fused GE2E loss fwd+bwd, microseconds per call (device time, CUDA-graph replay of the C-ABI call)", "unit": "us",
                      "higher_is_better": False, "n_gpus": 1, "data": "synthetic", "dtype": "f32 (N < 256) / split-fp16 tensor core",
                      "config": {"workload": "ge2e_sweep_N64-4096_M15_D256"}, "peaks": pk, "sweep": rows}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="train workload: after the timed steps, write what the last one computed (loss, d-vectors, "
                         "updated parameters and their gradients, ~21 MB) as DIR/<name>.npy in float32; the inputs "
                         "depend only on the arguments, so two builds can be compared output for output.  Weight "
                         "gradients are summed with fp32 atomics, so two runs of one build already differ by rounding "
                         "(and the few ReLU gates it flips): ~1e-6 in the loss, up to a few 1e-3 relative per gradient")
    ap.add_argument("--workload", default="train", choices=["train", "infer", "ge2e"],
                    help="train: GE2E training step (headline, BASELINE config 2/4, the line also carries config 3); "
                         "infer: multi-slice extraction alone (config 3); ge2e: fused-loss sweep (config 5)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "native" or args.workload != "train"):
        ap.error("--dump-outputs writes the outputs of the native train workload only")
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "infer":
        run_infer(args)
    elif args.workload == "ge2e":
        run_ge2e(args)
    else:
        run_native(args)


if __name__ == "__main__":
    main()
