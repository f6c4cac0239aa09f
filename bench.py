#!/usr/bin/env python
"""bench.py — VampNet masked-token generation hot path on B200 (contract in the task statement).

    python bench.py --gpus N --steps K --warmup W [--config {1,2,3,4}]     # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K --warmup W         # CPU arm (oracle port of the reference)
    torchrun ... bench.py --gpus N ...                                     # N>1: one rank per GPU, weak scaling

--config selects BASELINE.json configs[k] (default 2, the configuration the metric "coarse+c2f" is quoted on):
  1  coarse generate: 12 sampling steps, T=768, B=8 per GPU
  2  coarse -> c2f full vamp: 12 + 24 steps, codebooks 4 -> 14, T=768, B=32 per GPU, unchunked
  3  DAC encode -> vamp -> DAC decode end to end through Interface, 10 s 44.1 kHz clips (T=575), 32 clips per GPU
     (256 over 8 GPUs), coarse 12 + c2f 24 steps; `value` has the audio resident in HBM, `e2e` host audio in / out
  4  long-context coarse: T=3072 (~40 s), 24 steps, B=8 per GPU (64 over 8 GPUs)
One "step" = one pass of that workload over one batch of synthetic input (random-init weights, random codes /
synthetic audio, periodic prompt every 7th frame, default sampling parameters: temperature 1, mask_temperature 10.5).
value = codec tokens/s = N*B*T*C_out / time (C_out = 4 for the coarse-only configs, 14 otherwise); real-time factor
= N*B*T*768/44100 / time.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

COARSE = dict(n_heads=20, n_layers=20, n_codebooks=4, n_conditioning_codebooks=0, embedding_dim=1280)
C2F = dict(n_heads=20, n_layers=16, n_codebooks=14, n_conditioning_codebooks=4, embedding_dim=1280)
HOP, SR = 768, 44100
CONFIGS = {
    1: dict(B=8, T=768, stages=(("coarse", 12),), c_out=4, codec=False,
            metric="codec tokens/sec (coarse generate 12 steps, T=768, 44.1 kHz)",
            workload="BASELINE.json configs[1]: coarse generate 12 steps (4 codebooks, 20 layers, d=1280), default sampling"),
    2: dict(B=32, T=768, stages=(("coarse", 12), ("c2f", 24)), c_out=14, codec=False,
            metric="codec tokens/sec (coarse 12 steps + c2f 24 steps generate, T=768, 44.1 kHz)",
            workload="BASELINE.json configs[2]: coarse generate 12 steps (4 codebooks, 20 layers) -> c2f "
                     "generate 24 steps (14 codebooks, 16 layers), unchunked, d=1280, default sampling"),
    3: dict(B=32, T=575, stages=(("coarse", 12), ("c2f", 24)), c_out=14, codec=True,
            metric="codec tokens/sec (DAC encode -> coarse 12 + c2f 24 steps -> DAC decode, 10 s clips, 44.1 kHz)",
            workload="BASELINE.json configs[3]: Interface.encode -> coarse_vamp (12 steps) -> coarse_to_fine (24 steps, "
                     "unchunked) -> Interface.decode on 10 s 44.1 kHz clips (441 000 samples -> 575 frames); codec = "
                     "DAC-family stand-in (lac is not available), tensor-core path"),
    4: dict(B=8, T=3072, stages=(("coarse", 24),), c_out=4, codec=False,
            metric="codec tokens/sec (long-context coarse generate 24 steps, T=3072, 44.1 kHz)",
            workload="BASELINE.json configs[4]: coarse generate 24 steps, T=3072 (~40 s), d=1280, 20 layers"),
}
MODEL_CFG = {"coarse": COARSE, "c2f": C2F}
# codec algorithmic work per 10 s clip (SURVEY.md section 8d, stand-in configuration): fp32 layer-by-layer bytes, flops
CODEC_BYTES = {"encode": 8.3e9, "decode": 12.4e9}
CODEC_FLOPS = {"encode": 0.61e12, "decode": 1.37e12}


def fwd_flops(cfg, T):
    """Algorithmic FLOPs of one sequence-forward (SURVEY.md §8d): T*[L*(20d^2 + 4Td) + 2*(8C)*d + 2*d*V*Cp]."""
    d, L, Cn = cfg["embedding_dim"], cfg["n_layers"], cfg["n_codebooks"]
    Cp = Cn - cfg["n_conditioning_codebooks"]
    return T * (L * (20 * d * d + 4 * T * d) + 2 * 8 * Cn * d + 2 * d * 1024 * Cp)


def family_flops(cfg, T, B, steps):
    d, L, Cn = cfg["embedding_dim"], cfg["n_layers"], cfg["n_codebooks"]
    Cp = Cn - cfg["n_conditioning_codebooks"]
    M = B * T
    per = {
        "gemm_qkv": 2 * M * 3 * d * d * L, "gemm_attn_out": 2 * M * d * d * L, "gemm_ffn_up": 2 * M * 4 * d * d * L,
        "gemm_ffn_down": 2 * M * 2 * d * d * L, "gemm_classifier": 2 * M * d * 1024 * Cp,
        "attention": 4 * B * T * T * d * L,
    }
    return {k: v * steps for k, v in per.items()}


def gemm_algorithmic_bytes(B, T, d=1280):
    """Mean algorithmic HBM bytes of one GEMM launch of a layer (qkv, attn-out, ffn-up, ffn-down weighted 1:1:1:1):
    A + W + outputs read/written once (bf16 = 2 B, fp32 residual = 4 B read + 4 B written + 2 B bf16 copy)."""
    M = B * T
    qkv = M * d * 2 + 3 * d * d * 2 + M * 3 * d * 2
    out = M * d * 2 + d * d * 2 + M * d * (4 + 4 + 2)
    up = M * d * 2 + 4 * d * d * 2 + M * 2 * d * 2
    down = M * 2 * d * 2 + 2 * d * d * 2 + M * d * (4 + 4 + 2)
    return (qkv + out + up + down) / 4.0


def ncu_traffic_per_launch():
    """dram__bytes_read.sum + dram__bytes_write.sum per GEMM launch from the committed `ncu --set full` summary
    (profiles/ncu_layer_r2.txt: one layer's qkv / attn-out / ffn-up / ffn-down at the bench shape)."""
    name = next((n for n in ("ncu_layer_r2.txt", "ncu_gemm_r1_pair.txt", "ncu_gemm_r1_final.txt")
                 if os.path.exists(os.path.join(ROOT, "profiles", n))), "ncu_layer_r2.txt")
    path = os.path.join(ROOT, "profiles", name)
    try:
        per_kind, cur = {}, None
        for line in open(path):
            if line.startswith("== "):
                cur = line.split("gemm_tcgen05_kernel<")[1][0] if "gemm_tcgen05_kernel<" in line else None
                if cur is not None:
                    per_kind.setdefault(cur, []).append(0.0)
            elif cur is not None and ("dram__bytes_read.sum " in line or "dram__bytes_write.sum " in line):
                f = line.split()
                val, unit = float(f[1]), f[2].lower()
                per_kind[cur][-1] += val * {"byte": 1.0, "kbyte": 1e3, "mbyte": 1e6, "gbyte": 1e9}[unit]
        # <1> qkv, <2> residual epilogue (attn-out and ffn-down alternate), <3> ffn-up: weight 1 : 2 : 1
        if not all(k in per_kind for k in "123"):
            return None, f"profiles/{name} incomplete"
        mean = lambda v: sum(v) / len(v)
        return (mean(per_kind["1"]) + 2 * mean(per_kind["2"]) + mean(per_kind["3"])) / 4.0, \
            f"profiles/{name} (ncu --set full, B=32 T=768 coarse layer)"
    except Exception as e:  # the summary is evidence, not a dependency
        return None, f"unavailable: {e}"


# ----------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows = []
        self.proc = None
        self.index = index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------------- CPU arm
def host_threads():
    """Threads the process may actually use: min(os.cpu_count(), affinity, cgroup cpu.max quota).  The GPU boxes
    report 128 logical CPUs but cap the container at 16 (cpu.max 1600000/100000); 128 torch threads on a
    16-CPU quota run ~15x slower than 16 threads."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = min(n, max(1, int(int(q) / int(per))))
    except Exception:
        pass
    return n


def cpu_sample(threads, cfg):
    """Bounded sample of the same workload on the host cores through the oracle port of the reference
    (oracle/vampnet_oracle.py, fp32 like the reference's CPU path): ONE sampling iteration (forward + sample + remask)
    of every stage at B=1 and the config's T, extrapolated to the config's iteration counts per clip; for the
    end-to-end config also one encode + decode of one clip through the codec oracle.  The port leaves out work the
    reference does and discards (typical_filter, transformer.py:989-993: ~30 % of its sampling time, BASELINE.md section 2),
    so the unmodified reference is somewhat SLOWER than this number."""
    from oracle import vampnet_oracle as vo
    torch.set_num_threads(threads)
    res = {}
    g = torch.Generator().manual_seed(0)
    T = cfg["T"]
    for tag, steps in cfg["stages"]:
        ocfg = vo.OracleConfig(**MODEL_CFG[tag])
        sd = vo.make_state_dict(ocfg, seed=0)
        orc = vo.OracleVampNet(ocfg, sd, "fp32")
        cb = vo.make_codebooks(ocfg.n_codebooks, seed=1)
        z = torch.randint(0, 1024, (1, ocfg.n_codebooks, T), generator=g)
        mask = torch.ones_like(z)
        mask[:, :, ::7] = 0
        mask[:, :ocfg.n_conditioning_codebooks] = 0
        t0 = time.perf_counter()
        orc.generate(cb, z, mask, _sampling_steps=1, seed=0, rng="torch")
        res[tag] = time.perf_counter() - t0
        del orc, sd
    clip_s = sum(steps * res[tag] for tag, steps in cfg["stages"])
    if cfg["codec"]:
        from oracle import dac_oracle as do
        ccfg = do.CodecConfig()
        w = do.make_codec_weights(ccfg, seed=0)
        x = 0.3 * torch.randn(1, 1, T * HOP, generator=g)
        t0 = time.perf_counter()
        with torch.no_grad():
            enc = do.encode(x, w, ccfg)
            do.decode(enc["z"], w, ccfg)
        res["codec"] = time.perf_counter() - t0
        clip_s += res["codec"]
    return T * cfg["c_out"] / clip_s, res


def cpu_sample_text(cfg, parts, threads):
    it = " + ".join(f"1 {tag} sampling iteration ({parts[tag]:.2f}s)" for tag, _ in cfg["stages"])
    ex = "+".join(str(n) for _, n in cfg["stages"])
    codec = f" + one codec-oracle encode/decode of a 10 s clip ({parts['codec']:.1f}s)" if cfg["codec"] else ""
    return (f"{it} at B=1,T={cfg['T']} via the oracle port (fp32, {threads} threads), extrapolated to {ex} iterations "
            f"per clip{codec}; the port omits the reference's discarded typical_filter work, so the unmodified "
            f"reference is slower than this")


def run_reference_arm(args, rank):
    if rank != 0:
        return
    cfg = CONFIGS[args.config]
    threads = host_threads()
    vals = []
    for i in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        v, parts = cpu_sample(threads, cfg)
        dt = time.perf_counter() - t0
        if i >= args.warmup:
            vals.append((v, dt))
    v = statistics.mean(x[0] for x in vals)
    line = {
        "metric": cfg["metric"], "value": v, "unit": "tokens/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * statistics.mean(x[1] for x in vals), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "impl": "reference",
        "rtf": v / cfg["c_out"] * HOP / SR,
        "config": {"workload": cfg["workload"] + "; bounded CPU sample at B=1", "seq_len": cfg["T"], "global_batch": 1},
        "cpu_baseline": {"value": v, "unit": "tokens/s", "cores": threads, "kind": "port",
                         "sample": "per step: " + cpu_sample_text(cfg, parts, threads)},
        "e2e": {"value": v, "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ----------------------------------------------------------------------------------------------- GPU arm
class _Codec:
    def __init__(self, cb):
        import types
        self.quantizer = types.SimpleNamespace(quantizers=[types.SimpleNamespace(
            codebook=types.SimpleNamespace(weight=cb[i])) for i in range(cb.shape[0])])
        self.sample_rate, self.hop_length = SR, HOP


def broadcast_weights(models, world):
    """NCCL over NVLink: rank 0's weights to every rank, one flat blob per model (the only collective on this path)."""
    if world == 1:
        return
    from vampnet_b200.parallel import broadcast_module_weights
    broadcast_module_weights(models, src=0)


_REAL_STDOUT = None


def quiet_stdout():
    """The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints its version banner from C),
    so fd 1 is pointed at stderr for the whole run and the JSON line is written to the saved descriptor."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line: dict):
    data = (json.dumps(line) + "\n").encode()
    sys.stdout.flush()
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, data)


def secondary_rooflines(cfg, B, fam_ms, fam_n, fl, peaks, codec_ms):
    """The kernels the north-star classifies by HBM bandwidth, and attention by tensor throughput, next to the headline
    GEMM family: achieved = ALGORITHMIC bytes (or flops) of the launches of one profiled step / their CUDA-event time."""
    hbm = peaks.get("hbm_gbs", 6650.0)
    tf = peaks.get("bf16_tflops_sustained", 1400.0)
    out = []
    T = cfg["T"]
    logit_bytes = emb_bytes = 0.0
    for tag, steps in cfg["stages"]:
        m = MODEL_CFG[tag]
        Cn, Cp, d = m["n_codebooks"], m["n_codebooks"] - m["n_conditioning_codebooks"], m["embedding_dim"]
        logit_bytes += steps * B * T * Cp * 1024 * 4.0                        # fp32 logits read once per iteration
        emb_bytes += steps * B * T * (Cn * (4 + 32) + d * (4 + 2) + 8)        # codes + table rows in, x fp32 + bf16 copy out
    if fam_ms.get("sample_remask"):
        from vampnet_b200 import _lib
        import ctypes
        v = ctypes.c_int32(0)
        _lib.lib().vnb_get_option(b"fused_sampler", ctypes.byref(v))
        if v.value:
            # the sampling sweeps run in the classifier GEMM's epilogue (counted under gemm_classifier); what is left
            # here reads 16 bytes per (position, 128-entry vocabulary tile) and writes token + confidence
            rec_bytes = logit_bytes / (128 * 4.0) * 16.0 + logit_bytes / (1024 * 4.0) * 12.0
            a = rec_bytes / (fam_ms["sample_remask"] * 1e-3) / 1e9
            out.append({"kernel": "sample_combine_kernel + remask_kernel (sampler fused into the classifier epilogue)",
                        "bound": "hbm", "achieved": a, "peak": hbm, "unit": "GB/s", "frac": a / hbm,
                        "algorithmic_bytes_per_step": rec_bytes, "ms_per_step": fam_ms["sample_remask"],
                        "logit_bytes_not_moved_per_step": 2 * logit_bytes,
                        "note": "latency-bound tail of the fused sampler: the fp32 logits (written and read once per "
                                "iteration before) no longer reach HBM; one thread per position, 4-pass radix select per clip"})
        else:
            a = logit_bytes / (fam_ms["sample_remask"] * 1e-3) / 1e9
            out.append({"kernel": "sample_rows_kernel + remask_kernel", "bound": "hbm", "achieved": a, "peak": hbm, "unit": "GB/s",
                        "frac": a / hbm, "algorithmic_bytes_per_step": logit_bytes, "ms_per_step": fam_ms["sample_remask"],
                        "note": "contract figure: every fp32 logit read once (SURVEY.md 8d); positions already known are "
                                "skipped by the kernel, so the bytes actually moved are fewer"})
    if fam_ms.get("embed"):
        a = emb_bytes / (fam_ms["embed"] * 1e-3) / 1e9
        out.append({"kernel": "embed (codes -> residual stream)", "bound": "hbm", "achieved": a, "peak": hbm, "unit": "GB/s",
                    "frac": a / hbm, "algorithmic_bytes_per_step": emb_bytes, "ms_per_step": fam_ms["embed"]})
    if fam_ms.get("attention"):
        a = fl["attention"] / (fam_ms["attention"] * 1e-3) / 1e12
        out.append({"kernel": "attention_tcgen05_kernel", "bound": "tensor", "achieved": a, "peak": tf, "unit": "TFLOP/s",
                    "frac": a / tf, "ms_per_step": fam_ms["attention"],
                    "note": "at d_head 64 the exponentials (MUFU) cost twice the tensor cycles: MUFU-bound ceiling = 0.5"})
    for part in ("encode", "decode"):
        if codec_ms.get(part):
            t = codec_ms[part] * 1e-3
            ab, af = B * CODEC_BYTES[part] / t / 1e9, B * CODEC_FLOPS[part] / t / 1e12
            out.append({"kernel": f"codec {part} (conv_tcgen05_kernel stack + rvq_kernel)", "bound": "hbm",
                        "achieved": ab, "peak": hbm, "unit": "GB/s", "frac": ab / hbm, "ms_per_step": codec_ms[part],
                        "tflops": af, "tensor_frac_of_sustained_bf16": af / tf,
                        "note": "bytes = fp32 layer-by-layer activation traffic of the stand-in architecture (SURVEY.md 8d); "
                                "split-bf16 issues 3 MMAs per algorithmic one"})
    return out


DUMP_BUDGET = 64_000_000  # bytes, .npy headers included


def dump_outputs(out_dir, arrays):
    """Write each tensor as out_dir/<name>.npy (float32).  When the total exceeds DUMP_BUDGET every array is cut to
    its share by a fixed, seeded choice of flat indices (sorted), so two runs with the same arguments store the same
    elements."""
    os.makedirs(out_dir, exist_ok=True)
    total = sum(t.numel() * 4 for t in arrays.values())
    budget = DUMP_BUDGET - 4096 * len(arrays)
    for name, t in arrays.items():
        a = t.numpy().astype(np.float32, copy=False)
        if total > budget:
            keep = a.size * budget // total
            idx = np.sort(np.random.default_rng(0).choice(a.size, size=keep, replace=False))
            a = a.reshape(-1)[idx]
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def main():
    quiet_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=sorted(CONFIGS), help="BASELINE.json configs[k]")
    ap.add_argument("--batch", type=int, default=None, help="clips per GPU (default = the named config)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned (rank 0) to DIR/<name>.npy, float32, "
                         f"at most {DUMP_BUDGET // 10**6} MB in all")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "b200":
        ap.error("--dump-outputs records the b200 path's outputs")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    cfg = CONFIGS[args.config]

    if args.impl == "reference":
        run_reference_arm(args, rank)
        return

    if args.warmup < 3:
        args.warmup = 3
    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback on the product path)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    from vampnet_b200 import _lib
    from vampnet_b200.modules.transformer import VampNet

    lib = _lib.lib()
    torch.manual_seed(1234)
    stage_names = [tag for tag, _ in cfg["stages"]]
    steps_of = dict(cfg["stages"])
    with torch.device(dev):
        models = {tag: VampNet(**MODEL_CFG[tag]) for tag in stage_names}
        cb = torch.randn(14, 1024, 8)
    to_bcast = list(models.values())
    iface = None
    if cfg["codec"]:
        from vampnet_b200.codec import DAC
        from vampnet_b200.interface import Interface
        dac = DAC()
        iface = Interface.from_models(dac, models["coarse"], models["c2f"], device=dev, coarse_chunk_size_s=10,
                                      coarse2fine_chunk_size_s=10)   # s2t(10) = 575 frames: one chunk per clip
        to_bcast.append(dac)
    broadcast_weights(to_bcast, world)
    if world > 1:
        dist.broadcast(cb, src=0)
    codec = iface.codec if iface is not None else _Codec(cb)

    B, T = (args.batch or cfg["B"]), cfg["T"]
    g = torch.Generator().manual_seed(100 + rank)  # every rank vamps its own clips

    def generate_stages(z, mask, mask_c2f, seed):
        zc = models["coarse"].generate(codec, start_tokens=z[:, :4].contiguous(), mask=mask[:, :4].contiguous(),
                                       _sampling_steps=steps_of["coarse"], return_signal=False, seed=seed)
        if "c2f" not in models:
            return zc
        zin = torch.cat([zc, z[:, 4:]], dim=1)
        return models["c2f"].generate(codec, start_tokens=zin, mask=mask_c2f, _sampling_steps=steps_of["c2f"],
                                      return_signal=False, seed=seed + 1)

    codec_ms = {}
    if not cfg["codec"]:
        z_host = torch.randint(0, 1024, (B, 14, T), generator=g).pin_memory()
        mask_host = torch.ones(B, 14, T, dtype=torch.int64)
        mask_host[:, :, ::7] = 0
        mask_host = mask_host.pin_memory()
        z_dev, mask_dev = z_host.to(dev), mask_host.to(dev)
        mask_c2f_dev = mask_dev.clone()
        mask_c2f_dev[:, :4] = 0  # conditioning codebooks are never masked (interface.py:355-357)

        def step_dev(seed):
            return generate_stages(z_dev, mask_dev, mask_c2f_dev, seed)

        def step_e2e(seed):
            zd = z_host.to(dev, non_blocking=True)
            md = mask_host.to(dev, non_blocking=True)
            mc = md.clone()
            mc[:, :4] = 0
            return generate_stages(zd, md, mc, seed).cpu()

        h2d = z_host.numel() * 8 + mask_host.numel() * 8
        api = " -> ".join(f"VampNet.generate({t})" for t in stage_names) + " with pinned host tensors in, host tensor out"
    else:
        from vampnet_b200.audio import AudioSignal
        n = 441000
        t = torch.arange(n) / SR
        f0 = 110.0 + 20.0 * torch.arange(B)[:, None] + 7.0 * rank
        clips_host = (0.3 * torch.sin(2 * torch.pi * f0 * t[None, :]) + 0.05 * torch.randn(B, n, generator=g))[:, None, :]
        clips_host = clips_host.contiguous().pin_memory()
        clips_dev = clips_host.to(dev)

        def pipeline(audio_dev, seed, timed=None):
            """Interface.encode -> build_mask -> coarse_vamp -> coarse_to_fine -> decode (reference interface.py:220,
            454, 383, 328, 203); `timed` collects CUDA-event times of the codec halves."""
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)] if timed is not None else None
            if ev:
                ev[0].record()
            codes = iface.encode(AudioSignal(audio_dev, SR))                   # (B, 14, 575)
            if ev:
                ev[1].record()
            mask = iface.build_mask(codes, None, periodic_prompt=7, upper_codebook_mask=3)
            zc = iface.coarse_vamp(codes, mask, _sampling_steps=steps_of["coarse"], seed=seed)
            z = iface.coarse_to_fine(zc, mask=mask, _sampling_steps=steps_of["c2f"], seed=seed + 1)
            if ev:
                ev[2].record()
            out = iface.decode(z)
            if ev:
                ev[3].record()
                torch.cuda.synchronize()
                timed["encode"], timed["decode"] = ev[0].elapsed_time(ev[1]), ev[2].elapsed_time(ev[3])
            return out.samples

        def step_dev(seed):
            return pipeline(clips_dev, seed)

        def step_e2e(seed):
            return pipeline(clips_host.to(dev, non_blocking=True), seed).cpu()

        h2d = clips_host.numel() * 4
        api = ("Interface.encode -> build_mask -> coarse_vamp -> coarse_to_fine -> Interface.decode with pinned host "
               "audio in, host audio out")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(args.warmup):
        out = step_dev(10 + 2 * i)
    torch.cuda.synchronize()
    if not cfg["codec"]:
        assert not (out == 1024).any(), "mask tokens survived generate()"
    else:
        assert out.shape == (B, 1, 441600) and bool(torch.isfinite(out).all())

    # ---- timed region: inputs resident in HBM, production path (CUDA-graph replay) ----
    clocks = ClockSampler(local_rank)
    clocks.start()
    time.sleep(0.3)
    launches0 = lib.vnb_launch_count()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        out = step_dev(100 + 2 * i)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    launches = lib.vnb_launch_count() - launches0
    clk = clocks.stop()
    # copied now: later calls may reuse the buffers the last timed step returned
    dumped = {("audio" if cfg["codec"] else "tokens"): out.float().cpu()} if args.dump_outputs and rank == 0 else None

    # ---- end to end: host (pinned) inputs, H2D + D2H inside the timed region, public API ----
    barrier()
    t0 = time.perf_counter()
    for i in range(args.steps):
        res_host = step_e2e(200 + 2 * i)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    barrier()
    d2h = res_host.numel() * res_host.element_size()

    # max over ranks
    tms = torch.tensor([ms, e2e_s * 1e3], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
    ms, e2e_ms = tms.tolist()

    # ---- per-kernel-family device time (CUDA events around every launch; graph bypassed) ----
    fam_ms = {k: 0.0 for k in _lib.FAMILIES}
    fam_n = {k: 0 for k in _lib.FAMILIES}
    fl = {}
    for tag in stage_names:
        for k, v in family_flops(MODEL_CFG[tag], T, B, steps_of[tag]).items():
            fl[k] = fl.get(k, 0) + v
    for model in models.values():
        _lib.check(lib.vnb_profile_begin(model._handle))
    if cfg["codec"]:
        pipeline(clips_dev, 300, timed=codec_ms)
    else:
        step_dev(300)
    torch.cuda.synchronize()
    for model in models.values():
        a = (C.c_float * len(_lib.FAMILIES))()
        n = (C.c_int32 * len(_lib.FAMILIES))()
        _lib.check(lib.vnb_profile_end(model._handle, a, n, len(_lib.FAMILIES)))
        for i, k in enumerate(_lib.FAMILIES):
            fam_ms[k] += a[i]
            fam_n[k] += n[i]
    prof_total = sum(fam_ms.values()) + sum(codec_ms.values())
    gemm_keys = [k for k in _lib.FAMILIES if k.startswith("gemm")]
    gemm_ms = sum(fam_ms[k] for k in gemm_keys)
    gemm_fl = sum(fl[k] for k in gemm_keys)
    gemm_n = sum(fam_n[k] for k in gemm_keys)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak_tf = peaks.get("bf16_tflops_sustained", 1400.0)  # kernel timed inside a long step -> sustained figure
    traffic, traffic_note = ncu_traffic_per_launch()
    if (B, T) != (32, 768):
        traffic, traffic_note = None, "the committed ncu capture is of the B=32, T=768 shape"
    achieved = gemm_fl / (gemm_ms * 1e-3) / 1e12 if gemm_ms > 0 else 0.0
    roofline = {
        "kernel": "gemm_tcgen05_kernel<EPI, PAIR=true> (CTA pairs, tcgen05.mma.cta_group::2, 256x256 tiles; all epilogues: qkv, attn-out+residual, ffn-up+GEGLU, ffn-down+residual, classifier+bias)",
        "bound": "tensor", "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved / peak_tf,
        "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained" if peaks else "fallback 1.4 PFLOP/s sustained",
        "traffic": traffic, "traffic_unit": "bytes per launch (dram read+write)", "traffic_source": traffic_note,
        "algorithmic_bytes_per_launch": gemm_algorithmic_bytes(B, T),
        "flops_per_launch": gemm_fl / max(gemm_n, 1), "avg_launch_us": 1e3 * gemm_ms / max(gemm_n, 1),
        "share_of_step": gemm_ms / prof_total if prof_total else None,
        "breakdown_ms": {**{k: round(fam_ms[k], 3) for k in _lib.FAMILIES}, **{"codec_" + k: round(v, 3) for k, v in codec_ms.items()}},
        "breakdown_tflops": {k: (fl[k] / (fam_ms[k] * 1e-3) / 1e12 if fam_ms.get(k) else None) for k in fl},
        "profiled_step_ms": prof_total,
        "secondary": secondary_rooflines(cfg, B, fam_ms, fam_n, fl, peaks, codec_ms),
    }

    if rank == 0:
        tokens = world * B * T * cfg["c_out"] * args.steps
        value = tokens / (ms * 1e-3)
        flops_step = sum(fwd_flops(MODEL_CFG[tag], T) * steps_of[tag] for tag in stage_names) * B
        if cfg["codec"]:
            flops_step += B * (CODEC_FLOPS["encode"] + CODEC_FLOPS["decode"])
        line = {
            "metric": cfg["metric"], "value": value, "unit": "tokens/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "rtf": world * B * T * HOP / SR * args.steps / (ms * 1e-3),
            "tflops": world * flops_step * args.steps / (ms * 1e-3) / 1e12,
            "config": {"workload": cfg["workload"], "baseline_config_index": args.config,
                       "global_batch": world * B, "per_gpu_batch": B, "seq_len": T, "parallelism": f"dp{world} (clips)",
                       "l2": "working set per step (1.3-2.4 GB of bf16 weights, plus ~1 GB of activations per layer) far exceeds the 126 MB L2",
                       "weights": "random-init, NCCL-broadcast from rank 0", "cuda_graph": True},
            "clocks": clk,
            "e2e": {"value": tokens / (e2e_ms * 1e-3), "unit": "tokens/s", "h2d_bytes_per_step": h2d * world,
                    "d2h_bytes_per_step": d2h * world, "ms_per_step": e2e_ms / args.steps, "api": api,
                    "rtf": world * B * T * HOP / SR * args.steps / (e2e_ms * 1e-3)},
            "gpu_launches": int(launches),
            "roofline": roofline,
        }
        if world == 1 and not args.no_cpu_baseline:
            threads = host_threads()
            v, parts = cpu_sample(threads, cfg)
            line["cpu_baseline"] = {"value": v, "unit": "tokens/s", "cores": threads, "kind": "port",
                                    "sample": cpu_sample_text(cfg, parts, threads)}
        emit(line)
        if dumped is not None:
            dump_outputs(args.dump_outputs, dumped)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
