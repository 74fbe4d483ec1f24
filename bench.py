#!/usr/bin/env python3
"""bench.py — ZKAttest proofs/s on B200 (contract in the task brief, tier section 4).

  python bench.py [--gpus N] [--steps K] [--warmup W]             our arm (CUDA, libzkattest.so)
  python bench.py --impl reference [--gpus N] [--steps K] ...     CPU arm (oracle port on host cores)
  torchrun --nproc-per-node N bench.py --gpus N ...               one rank per GPU (weak scaling)

A "step" = one zka_prove_batch pass over one batch of synthetic signatures (per rank), followed,
for N > 1, by ONE NCCL all-gather of the serialized proof bytes (BASELINE.json north_star).
Workload at N=1: BASELINE.json configs[2] = batch 8192 proofs, ring N=256, the largest single-GPU
configuration; under torchrun (N>1): 8192 proofs per GPU, ring N=1024 = configs[3] (prove) and
configs[4] (verify) at 8 GPUs, weak scaling.  `--workload config1|config2|config3` overrides.
`value`  : proofs/s, inputs resident in HBM, device pointers through the C ABI.
`e2e`    : proofs/s through the same C-ABI call with pinned HOST buffers (H2D tape/inputs and
           D2H proofs inside the timed region).
`roofline`: dominant kernel (TomCommitTask) 32x32->64 multiply-accumulates per second against
           the measured IMAD.WIDE peak of this GPU (tools/imad_peak); HBM GB/s reported beside it.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (batch per GPU, ring size)   — BASELINE.json configs[1..3]
    'config1': (1024, 8),
    'config2': (8192, 256),
    'config3': (8192, 1024),   # 65536 / 8 GPUs
}
SEC_LEVEL = 80
# executed field multiplications per tomEdwards256 commitment: 2*nwin mixed additions x 8 modmul,
# each modmul = 9x9 product + 5 generic modulus limbs x 9 quotient digits = 126 32x32 MACs
# DRAM bytes per table lookup of the commitment kernels, from `ncu --set full` captures (profiles/):
# window bits -> (dram read + write bytes per launch - algorithmic bytes) / lookups
NCU_DRAM_BYTES_PER_LOOKUP = {16: 78.0, 22: 118.0}
# DRAM bytes per (entry, window) of the aggregate verify MSM (profiles/pipes_r2m_config2.md: 5.75 GB over two launches of
# 4096 proofs x ~373 entries x 18 windows); the algorithmic figure is a 128-byte entry + a 4-byte index
NCU_DRAM_BYTES_PER_AGG_ENTRY_WINDOW = 105.0
MODMUL_PER_MADD = 7      # a = -1 image curve, mixed addition with (v-w, v+w, 2 d2 w v) entries (zk_curves.cuh)
MAC_PER_TOM_MODMUL = 117   # EXECUTED IMAD.WIDE per 258-bit product: 9 rows x (9 + 4) (zk_field_ptx.cuh tom_row;
                           # profiles/sass_tom_mul_r2.txt); the generic CIOS needs 171
MAC_PER_P256_MODMUL = 64   # p256.p product scanning: 8 x 8, the reduction is additions only
MAC_PER_N256_MODMUL = 136  # p256.n generic CIOS: 64 + 64 + 8
W_PROVE_REF = {8: 6861088, 256: 6942368, 1024: 6974880}   # reference-algorithm modmuls/proof (SURVEY 8(d))
DUMP_BYTES = 60 << 20      # --dump-outputs: the arrays together; with the .npy headers all files stay below 64 MB


def dump_rows(B: int, row_bytes: int, fixed_bytes: int):
    """Rows of a (B, row_bytes) float32 array that fit in DUMP_BYTES beside `fixed_bytes`: all of them, or a fixed
    seeded sample in ascending order."""
    import numpy as np
    k = max(1, min(B, (DUMP_BYTES - fixed_bytes) // (4 * row_bytes)))
    return np.arange(B) if k == B else np.sort(np.random.default_rng(0).choice(B, k, replace=False))


def dump_outputs(out_dir: str, rows, proofs, proof_len, status, **extra):
    """Write what one prove call returned as float32 .npy files: the proof bytes of `rows` (zero past each proof's
    length, where the bytes are padding), every proof length and status, the row indices, and `extra` arrays."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    proofs = np.asarray(proofs).astype(np.float32)
    proofs[np.arange(proofs.shape[1])[None, :] >= np.asarray(proof_len)[rows][:, None]] = 0
    arrays = {'proofs': proofs, 'proof_rows': rows, 'proof_len': proof_len, 'status': status, **extra}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + '.npy'), np.asarray(a).astype(np.float32))


# ----------------------------------------------------------------------------------------- CPU arm
# The reference itself (TypeScript on node) cannot run in this image.  The CPU arm is oracle/cpu: a C++
# restatement of the reference's OWN algorithms (4-bit-window mul/dblmul, RCB / Hisil formulas, one inversion
# per toBytes, Bos-Coster verification) behind the same C ABI, byte-identical to the Python oracle and the
# golden fixtures (tests/test_cpu_port.py).  Native 64-bit-limb Montgomery code is several times faster than
# BigInt arithmetic in V8 would be, so ratios against it are conservative.
def usable_cores() -> int:
    """Host threads this process may actually use: affinity mask capped by the cgroup CPU quota."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    try:
        q, per = open('/sys/fs/cgroup/cpu.max').read().split()
        if q != 'max':
            n = max(1, min(n, int(int(q) / int(per))))
    except Exception:
        pass
    return n


class CpuPort:
    """oracle/_ref/libzkattest_cpu.so on `threads` host threads, fed with the synthetic workload of bench.py."""

    def __init__(self, N: int, threads: int):
        import numpy as np
        import __graft_entry__ as g
        from zkp_ecdsa_b200 import synth, verify_tape as VT
        from zkp_ecdsa_b200.capi import ZkaLib
        if not os.path.exists(g.ORACLE_CPU):
            g.build_oracle_cpu()
        os.environ['ZKA_CPU_THREADS'] = str(threads)
        self.np, self.N, self.threads = np, N, threads
        self.L = ZkaLib(g.ORACLE_CPU)
        hn, hp = self.L.params_generate(synth.params_rnd(0))
        self.P = self.L.params_create(hn, hp, SEC_LEVEL)
        self.synth, self.VT = synth, VT

    def sample(self, B: int, seed: int):
        np, L = self.np, self.L
        wl = self.synth.Workload(B, self.N, seed=seed, distinct_signers=min(B, self.N))
        tape = self.synth.random_tape(B, L.prove_tape_len(self.N, SEC_LEVEL), seed=seed + 1)
        vt = self.VT.random_verify_tape(B, L.verify_tape_len(self.N, SEC_LEVEL), self.N, SEC_LEVEL, seed=seed + 2)
        ps = L.proof_max_len(self.N, SEC_LEVEL)
        return wl, tape, vt, np.zeros((B, ps), np.uint8), np.zeros(B, np.uint32), np.zeros(B, np.int32), ps

    def prove(self, smp):
        wl, tape, vt, proofs, plen, st, ps = smp
        t = time.perf_counter()
        self.L.prove_batch(self.P, wl.B, wl.msg_hash, wl.sig, wl.pk, wl.which, wl.ring, self.N, tape, tape.shape[1], proofs, ps, plen, st)
        dt = time.perf_counter() - t
        assert not st.any(), st
        return dt

    def verify(self, smp):
        wl, tape, vt, proofs, plen, st, ps = smp
        ok = self.np.zeros(wl.B, self.np.uint8)
        t = time.perf_counter()
        self.L.verify_batch(self.P, wl.B, wl.msg_hash, wl.ring, self.N, proofs, ps, plen, vt, vt.shape[1], ok, st)
        dt = time.perf_counter() - t
        assert ok.all() and not st.any()
        return dt


def cpu_baseline(N: int, per_core: int = 2):
    """oracle/cpu on all usable host cores (threads inside one process), plus the single-thread figure."""
    cores = usable_cores()
    port = CpuPort(N, cores)
    smp = port.sample(cores * per_core, 1000)
    dt = port.prove(smp)
    dv = port.verify(smp)
    one = CpuPort(N, 1)
    s1 = one.sample(1, 2000)
    d1 = one.prove(s1)
    v1 = one.verify(s1)
    B = cores * per_core
    return {'value': B / dt, 'unit': 'proofs/s', 'cores': cores, 'kind': 'port-c++',
            'sample': f'{B} proofs (ring {N}, SecLevel {SEC_LEVEL}) on {cores} threads of oracle/cpu (C++ restatement of the '
                      f'reference algorithms; the TypeScript reference cannot run here: no node), {dt:.2f} s wall',
            'single_thread': {'value': 1.0 / d1, 'unit': 'proofs/s', 's_per_proof': d1},
            'verify': {'value': B / dv, 'unit': 'verifies/s', 'cores': cores, 'single_thread_s_per_verify': v1},
            'note': 'native Montgomery code on 64-bit limbs: several times faster than V8 BigInt would be, so GPU/CPU ratios '
                    'against it are conservative; the Python-int oracle (oracle/*.py) needs ~3 s per proof per core'}


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    wname = args.workload or ('config2' if args.gpus == 1 else 'config3')
    B, N = WORKLOADS[wname]
    cores = usable_cores()
    port = CpuPort(N, cores)
    for _ in range(min(args.warmup, 2)):
        port.prove(port.sample(cores, 3000))
    tot_s = 0.0
    tot_n = 0
    for k in range(args.steps):
        smp = port.sample(cores, 4000 + k)      # building the sample (keygen, signatures) is not timed
        tot_s += port.prove(smp)
        tot_n += cores
    if args.dump_outputs:
        _, _, _, proofs, plen, st, ps = smp
        rows = dump_rows(cores, ps, 3 * 4 * cores)
        dump_outputs(args.dump_outputs, rows, proofs[rows], plen, st)
    v = tot_n / tot_s
    line = {
        'impl': 'reference', 'metric': 'ZKAttest proofs/sec', 'value': v, 'unit': 'proofs/s',
        'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1e3 * tot_s / args.steps,
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'u256/u258 (64-bit limbs, Montgomery, C++)',
        'data': 'synthetic',
        'config': {'workload': f'{wname}: ring N={N}, SecLevel {SEC_LEVEL}; each step = a bounded sample of '
                               f'{cores} proofs (one per host thread) of the batch-{B} workload'},
        'cpu_baseline': {'value': v, 'unit': 'proofs/s', 'cores': cores, 'kind': 'port-c++',
                         'sample': f'{tot_n} proofs in {tot_s:.1f} s on {cores} threads of oracle/cpu (C++ restatement of the '
                                   'reference algorithms); the TypeScript reference itself cannot run here (no node)'},
        'e2e': {'value': v, 'unit': 'proofs/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    emit_json(line)


# ----------------------------------------------------------------------------------------- clocks
class ClockSampler:
    """SM clock / throttle-reason samples DURING the timed region: an NVML polling thread (every 5 ms;
    a timed region of a few steps is < 100 ms), `nvidia-smi -lms` as the fallback."""
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')
    REASON_BITS = {0x8: 'hw_slowdown', 0x40: 'hw_thermal_slowdown', 0x20: 'sw_thermal_slowdown', 0x4: 'sw_power_cap'}

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.samples = []          # (sm_mhz, max_mhz, power_w, reason_mask)
        self.proc = None
        self.nvml = None
        self.stop_flag = threading.Event()

    def _nvml_handle(self):
        import pynvml
        pynvml.nvmlInit()
        try:
            import torch
            uuid = str(torch.cuda.get_device_properties(self.idx).uuid)
            if not uuid.startswith('GPU-'):
                uuid = 'GPU-' + uuid
            return pynvml, pynvml.nvmlDeviceGetHandleByUUID(uuid)
        except Exception:
            return pynvml, pynvml.nvmlDeviceGetHandleByIndex(self.idx)

    def _sample(self, with_power=False):
        nv, h = self.nvml
        try:
            sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
            try:
                mask = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
            except Exception:
                mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
            pw = nv.nvmlDeviceGetPowerUsage(h) / 1000.0 if with_power else 0.0
            self.samples.append((float(sm), float(self.max_mhz), pw, int(mask)))
        except Exception:
            pass

    def _poll(self):
        # clock + event reasons only inside the loop (the power query is the slow one); every 5 ms
        k = 0
        while not self.stop_flag.wait(0.005):
            self._sample(with_power=(k % 8 == 0))
            k += 1

    def start(self):
        try:
            self.nvml = self._nvml_handle()
            self.max_mhz = self.nvml[0].nvmlDeviceGetMaxClockInfo(self.nvml[1], self.nvml[0].NVML_CLOCK_SM)
            self.th = threading.Thread(target=self._poll, daemon=True)
            self.th.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits',
                                          '-i', str(self.idx), '-lms', '100'], stdout=subprocess.PIPE, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            f = [x.strip() for x in line.strip().split(',')]
            if len(f) < 8:
                continue
            try:
                mask = 0
                for bit, v in zip((0x8, 0x40, 0x20, 0x4), f[4:8]):
                    if v.lower().startswith('active'):
                        mask |= bit
                self.samples.append((float(f[1]), float(f[2]), float(f[3]), mask))
            except ValueError:
                continue

    def stop(self):
        if self.nvml:
            self.stop_flag.set()
            self.th.join(timeout=2)
            if not self.samples:              # never happened so far; better a sample right after than none
                self._sample(with_power=True)
        elif self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        else:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['no NVML / nvidia-smi']}
        sm = sorted(x[0] for x in self.samples)
        reasons = set()
        for x in self.samples:
            for bit, name in self.REASON_BITS.items():
                if x[3] & bit:
                    reasons.add(name)
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': max((x[1] for x in self.samples), default=None),
                'power_w_max': max((x[2] for x in self.samples), default=None), 'samples': len(sm),
                'source': 'nvml' if self.nvml else 'nvidia-smi', 'reasons': sorted(reasons)}


# ----------------------------------------------------------------------------------------- our arm
def measured_int_peak(device_index: int):
    """IMAD.WIDE.U32 (32x32+64 MAC) peak of this GPU: live run of tools/imad_peak, else committed value."""
    exe = os.path.join(ROOT, 'tools', 'imad_peak')
    try:
        out = subprocess.run([exe], capture_output=True, text=True, timeout=60).stdout
        for ln in out.splitlines():
            d = json.loads(ln)
            if d.get('kernel') == 'imad_wide_u32_carry_chain':
                return d['gops'], 'measured live (tools/imad_peak, carry-chained IMAD.WIDE.U32)'
    except Exception:
        pass
    try:
        d = json.load(open(os.path.join(ROOT, 'profiles', 'imad_peak_b200.json')))
        return d['imad_wide_u32_carry_chain_gops'], 'profiles/imad_peak_b200.json (measured on this pool)'
    except Exception:
        return 9000.0, 'fallback 9.0e12/s (31 IMAD.WIDE/clk/SM x 148 SM x 1.965 GHz)'


def executed_mac_model(cfg, n_ring_bits, g_w=20, h_w=20):
    """EXECUTED 32x32+64 multiply-accumulates per work item of the kernels that hold the arithmetic
    (DESIGN.md 5).  Kernels not listed (hashing, byte assembly, layout, key dedup, the doubling chains of the
    few distinct keys) are counted as ZERO, so the whole-step figure is a lower bound of the utilisation."""
    T, P, Nn = MAC_PER_TOM_MODMUL, MAC_PER_P256_MODMUL, MAC_PER_N256_MODMUL
    nwin = cfg['tom_nwin']
    p256_madd = 13        # RCB15 Alg. 5: 11 M + 2 multiplications by b
    p256_add, p256_dbl = 14, 13
    pa_lookups = -(-256 // g_w) + -(-256 // h_w) + 52 * 31 / 32     # G table + h table + signed 5-bit pk table
    return {
        'TomCommitHTask': nwin * MODMUL_PER_MADD * T,
        'TomCommitGTask': nwin * MODMUL_PER_MADD * T,
        'TomCommitTask': 2 * nwin * MODMUL_PER_MADD * T,
        'PhaseAAndRPointTask': 5 * Nn + pa_lookups * p256_madd * P,
        'TomNormTask': 11 * T,              # per point; the chunk's binary inversion is ALU work + 4 products
        'P256NormTask': 7 * P,
        'ItemScalarsTask': 55 * P,
        'PhaseBP256Task': p256_madd * P,
        'DerivedTask': 6 * (9 + 1) * T,     # six complete additions + from_affine products
        # verifier
        'MsmP256WindowTask': (21 * 15 / 16 * p256_madd + 30 * p256_add) * P,
        'VSampleP256Task': 52 * 31 / 32 * p256_madd * P,
        'VParseEntriesTask': 9 * T,
        'VDerivedTask': (6 * 10 + 4 * 7) * T,
    }


def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    from zkp_ecdsa_b200 import api, sharding, synth
    from zkp_ecdsa_b200 import verify_tape as VT

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        # NCCL's INFO log (rank/topology/NVLS lines the driver greps) goes to stderr: fd 1 is already routed
        # there by quiet_stdout(), so nothing has to be silenced to keep stdout to the one JSON line
        if os.environ.get('NCCL_DEBUG', '').upper() not in ('INFO', 'TRACE'):
            os.environ['NCCL_DEBUG'] = 'INFO'      # (the image presets a quieter level: only the version line appeared)
        os.environ.setdefault('NCCL_DEBUG_SUBSYS', 'INIT,ENV')
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    wname = args.workload or ('config2' if world == 1 else 'config3')
    B, N = WORKLOADS[wname]
    if args.batch:
        B = args.batch
    if args.ring:
        N = args.ring
    nbits = max(1, (N - 1).bit_length())

    eng = api.Engine(device=local)
    L = eng.lib
    params = eng.generate_params_list(SEC_LEVEL, rnd=synth.params_rnd(0))
    wl = synth.Workload(B, N, seed=100 + rank)
    ts = L.prove_tape_len(N, SEC_LEVEL)
    ps = (L.proof_max_len(N, SEC_LEVEL) + 15) & ~15     # 16-byte aligned rows (zka_proofs_pack moves uint4)
    tape_h = torch.from_numpy(synth.random_tape(B, ts, seed=200 + rank)).pin_memory()

    def pin(a):
        return torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    h = {'msg': pin(wl.msg_hash), 'sig': pin(wl.sig), 'pk': pin(wl.pk), 'which': pin(wl.which.view(np.uint8)),
         'ring': pin(wl.ring)}
    d = {k: v.to(dev) for k, v in h.items()}
    tape_d = tape_h.to(dev)
    proofs_d = torch.zeros((B, ps), dtype=torch.uint8, device=dev)
    plen_d = torch.zeros(B, dtype=torch.int32, device=dev)
    stat_d = torch.zeros(B, dtype=torch.int32, device=dev)
    proofs_h = torch.zeros((B, ps), dtype=torch.uint8).pin_memory()
    plen_h = torch.zeros(B, dtype=torch.int32).pin_memory()
    stat_h = torch.zeros(B, dtype=torch.int32).pin_memory()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)   # > 126 MB L2
    lib_stream = torch.cuda.ExternalStream(L.stream_ptr(), device=dev)
    # N > 1: the all-gather of the proof bytes (packed to their true lengths) overlaps proving.  --gather-mode
    #   pipeline (default): ONE prove call per step into one of two output buffer sets; the gather of step k is queued on a
    #             communication stream and runs while step k + 1 is proved; the timed region ends when the last gather has
    #             landed.  Whole-job throughput is what `value` reports; `gather.exposed_ms_per_step` is the part not hidden.
    #   serial:   the gather follows its step and is fully exposed (3.3 ms at 2 GPUs, ~7x that at 8).
    #   chunks:   one prove call; a second host thread queues the gather of every chunk the library reports complete
    #             (zka_set_progress), in chunk order — needs more chunks than lanes, and chunks of 1376 instead of 2752
    #             proofs cost 11 % of the 2-GPU throughput (profiles/README.md).
    #   groups:   --gather-groups G sub-batches proved by separate calls (each call ends with a full synchronisation of
    #             its lanes: two groups cost 6 %, four 20 %).
    gather = None
    gathers, outbufs = [], [(proofs_d, plen_d)]
    mode = args.gather_mode if world > 1 else 'none'
    if world > 1:
        if mode == 'groups':
            gather = sharding.ProofGather(L, world, rank, B, ps, N, SEC_LEVEL, dev, groups=max(1, args.gather_groups))
        elif mode == 'chunks':
            if args.gather_chunk > 0:
                L.set_option('chunk', args.gather_chunk)     # more chunks than lanes: the early ones overlap the later ones
            off = L.chunk_schedule(B, host_buffers=False)
            gather = sharding.ProofGather(L, world, rank, B, ps, N, SEC_LEVEL, dev, ranges=list(zip(off[:-1], off[1:])))
        else:
            nb = 2 if mode == 'pipeline' else 1
            gathers = [sharding.ProofGather(L, world, rank, B, ps, N, SEC_LEVEL, dev, ranges=[(0, B)]) for _ in range(nb)]
            gather = gathers[0]
            if nb == 2:
                outbufs.append((torch.zeros((B, ps), dtype=torch.uint8, device=dev), torch.zeros(B, dtype=torch.int32, device=dev)))
    step_no = [0]

    def prove_dev(b0, b1, out=None):
        pd, pl = out if out is not None else (proofs_d, plen_d)
        L.prove_batch(params.handle, b1 - b0, d['msg'][b0:].data_ptr(), d['sig'][b0:].data_ptr(), d['pk'][b0:].data_ptr(),
                      d['which'][4 * b0:].data_ptr(), d['ring'].data_ptr(), N, tape_d[b0:].data_ptr(), ts,
                      pd[b0:].data_ptr(), ps, pl[b0:].data_ptr(), stat_d[b0:].data_ptr())

    def step_device():
        if world == 1:
            prove_dev(0, B)
            return
        if mode == 'chunks':
            gather.prove_overlapped(lambda: prove_dev(0, B), proofs_d, plen_d)
            return
        if mode == 'groups':
            gather.begin()
            for (b0, b1) in gather.ranges:
                prove_dev(b0, b1)
                gather.submit(proofs_d, plen_d, b0, b1)
            gather.finish()
            return
        i = step_no[0] % len(gathers)
        step_no[0] += 1
        g = gathers[i]
        g.finish()                        # the gather that used this buffer set (two steps ago) has landed
        prove_dev(0, B, outbufs[i])
        g.begin()
        g.submit(outbufs[i][0], outbufs[i][1], 0, B)
        if mode == 'serial':
            g.finish()

    def drain():
        for g in gathers:
            g.finish()

    def step_host():
        L.prove_batch(params.handle, B, h['msg'].data_ptr(), h['sig'].data_ptr(), h['pk'].data_ptr(),
                      h['which'].data_ptr(), h['ring'].data_ptr(), N, tape_h.data_ptr(), ts,
                      proofs_h.data_ptr(), ps, plen_h.data_ptr(), stat_h.data_ptr())

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, end=None):
        barrier()
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record(lib_stream)
        for _ in range(steps):
            flush.zero_()            # evict L2 between steps (torch stream; tiny vs a step)
            torch.cuda.current_stream().synchronize()
            fn()
        if end:
            end()
        torch.cuda.synchronize()
        e1.record(lib_stream)
        e1.synchronize()
        wall = time.perf_counter() - t0
        barrier()
        dev_ms = e0.elapsed_time(e1)
        t = torch.tensor([max(wall * 1e3, dev_ms)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # warm-up (>= 3 steps: allocator growth, table pages, clocks)
    for _ in range(max(args.warmup, 3)):
        step_device()
    drain()
    torch.cuda.synchronize()
    assert int((stat_d != 0).sum().item()) == 0, 'prover reported per-proof errors'

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0 = L.launch_count()
    for g in gathers:
        g.exposed_ms = []
    ms_total = timed(step_device, args.steps, drain)
    launches = L.launch_count() - l0
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        # the output buffer set of the last timed step, read before the passes below prove into it again
        out_p, out_l = outbufs[(step_no[0] - 1) % len(outbufs)]
        rows = dump_rows(B, ps, 5 * 4 * B)
        dump = {'proofs': out_p[torch.from_numpy(rows).to(dev)].cpu().numpy(), 'proof_len': out_l.cpu().numpy(),
                'status': stat_d.cpu().numpy()}
    ms_step = ms_total / args.steps
    value = world * B / (ms_step * 1e-3)
    gather_info = None
    if gathers:
        last = (step_no[0] - 1) % len(gathers)
        for i in range(len(gathers)):
            info = gathers[i].check(outbufs[i][0], outbufs[i][1])
            if i == last:
                gather_info = info
        gather_info['mode'] = mode
        gather_info['exposed_ms_per_step'] = sum(sum(g.exposed_ms) for g in gathers) / args.steps   # host time spent waiting for gathers
        if len(gathers) == 2:      # both output sets hold the same proofs (same inputs, same tape)
            assert torch.equal(outbufs[0][1], outbufs[1][1])
    elif gather:
        gather_info = gather.check(proofs_d, plen_d)
        gather_info['mode'] = mode

    # per-kernel CUDA-event pairs on the launching streams: a separate, un-timed pass (the event pairs
    # serialise the lanes of a call, so they are kept out of the timed region)
    psteps = max(1, min(args.steps, 3))
    lanes_cfg = L.config().get('lanes', 1)
    L.set_option('lanes', 1)          # one lane: the event pairs of concurrent lanes would time each other's kernels
    L.profile_reset()
    L.set_profiling(True)
    for _ in range(psteps):
        flush.zero_()
        torch.cuda.synchronize()
        prove_dev(0, B)
    L.set_profiling(False)
    L.set_option('lanes', lanes_cfg)
    prof = L.profile()
    ms_prof_step = sum(e['ms'] for e in prof.values()) / psteps

    # ---- end to end through the C ABI with host buffers (H2D + D2H inside)
    for _ in range(2):
        step_host()
    esteps = max(1, min(args.steps, 5))
    e2e_ms = timed(step_host, esteps) / esteps
    assert int((stat_h != 0).sum().item()) == 0
    # bytes that cross PCIe per step: the small inputs; the tape as the library uploads it (two strided copies: the
    # 3 + 4S draws before the challenge, then the item / GK draws up to the longest proof — counted here with the
    # longest proof of the whole batch; ZKA_TAPE_SPLIT=0: the full stride); every proof row up to the longest proof
    # (rows are stride-padded; one 2-D copy per chunk), the lengths and statuses
    zmax = int(((plen_h.max().item() - (264 + 80 * 330 + 1 + 4 * nbits * 67 + (3 * nbits + 1) * 33)) // (3596 - 330)))
    tape_bytes = 32 * (3 + 4 * SEC_LEVEL + 40 * zmax + 5 * nbits) if os.environ.get('ZKA_TAPE_SPLIT', '1') != '0' else int(tape_h.shape[1])
    h2d = sum(int(v.numel()) for v in h.values()) + B * tape_bytes
    d2h = int(plen_h.max().item()) * B + 8 * B
    # the two arms must agree bit for bit (valid prefix of every row; bytes past proof_len are padding)
    col = torch.arange(ps, device=dev).unsqueeze(0)
    valid = col < plen_d.unsqueeze(1)
    same = bool(torch.equal(plen_h.to(dev), plen_d)) and bool(((proofs_h.to(dev) == proofs_d) | ~valid).all().item())
    del col, valid
    # cost of producing the randomness itself (outside the timed regions: the C ABI takes the tape as an input)
    t0 = time.perf_counter()
    api.synth_os_tape(64, ts, SEC_LEVEL)
    tape_gen_s_per_proof = (time.perf_counter() - t0) / 64

    # ---- verifySignatureList over the proofs just produced: device resident and end to end
    vts = L.verify_tape_len(N, SEC_LEVEL)
    vt_h = torch.from_numpy(VT.random_verify_tape(B, vts, N, SEC_LEVEL, seed=300 + rank)).pin_memory()
    vt_d = vt_h.to(dev)
    ok_d = torch.zeros(B, dtype=torch.uint8, device=dev)
    vst_d = torch.zeros(B, dtype=torch.int32, device=dev)
    ok_h = torch.zeros(B, dtype=torch.uint8).pin_memory()
    vst_h = torch.zeros(B, dtype=torch.int32).pin_memory()
    ok_all = torch.zeros(world * B, dtype=torch.uint8, device=dev)

    def verify_dev():
        L.verify_batch(params.handle, B, d['msg'].data_ptr(), d['ring'].data_ptr(), N, proofs_d.data_ptr(), ps,
                       plen_d.data_ptr(), vt_d.data_ptr(), vts, ok_d.data_ptr(), vst_d.data_ptr())
        if world > 1:   # configs[4]: the verdicts of all ranks on every rank
            dist.all_gather_into_tensor(ok_all, ok_d)

    def verify_host():
        L.verify_batch(params.handle, B, h['msg'].data_ptr(), h['ring'].data_ptr(), N, proofs_h.data_ptr(), ps,
                       plen_h.data_ptr(), vt_h.data_ptr(), vts, ok_h.data_ptr(), vst_h.data_ptr())
    for _ in range(2):
        verify_dev()
    vsteps = max(1, min(args.steps, 5))
    lv0 = L.launch_count()
    v_ms = timed(verify_dev, vsteps) / vsteps
    vlaunches = (L.launch_count() - lv0) // vsteps
    all_ok = bool((ok_d == 1).all().item()) and bool((vst_d == 0).all().item())
    if world > 1:
        all_ok = all_ok and bool((ok_all == 1).all().item())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, rows, dump['proofs'], dump['proof_len'], dump['status'],
                     verify_ok=ok_d.cpu().numpy(), verify_status=vst_d.cpu().numpy())
    L.set_option('lanes', 1)
    L.profile_reset()
    L.set_profiling(True)
    for _ in range(2):
        flush.zero_()
        torch.cuda.synchronize()
        L.verify_batch(params.handle, B, d['msg'].data_ptr(), d['ring'].data_ptr(), N, proofs_d.data_ptr(), ps,
                       plen_d.data_ptr(), vt_d.data_ptr(), vts, ok_d.data_ptr(), vst_d.data_ptr())
    L.set_profiling(False)
    L.set_option('lanes', lanes_cfg)
    vprof = L.profile()
    agg_c_prof = L.stat('agg_c') if hasattr(L, 'stat') else 0     # window bits of the aggregate MSM in the profiled pass
    ms_vprof_step = sum(e['ms'] for e in vprof.values()) / 2
    verify_host()
    ve2e_ms = timed(verify_host, vsteps) / vsteps
    v_e2e_ok = bool((ok_h == 1).all().item()) and bool((vst_h == 0).all().item())
    v_h2d = int(plen_h.sum().item()) if False else B * ps + B * (32 + 4 + vts) + N * 32
    zero_bits = ((plen_h.to(torch.int64) - (264 + 80 * 330 + 1 + 4 * nbits * 67 + (3 * nbits + 1) * 33)) // (3596 - 330)).float().mean().item()

    if world > 1:
        lt = torch.tensor([launches], dtype=torch.int64, device=dev)
        dist.all_reduce(lt)
        launches = int(lt.item())
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- rooflines: executed multiply-accumulates against the measured IMAD.WIDE peak of this GPU
    cfg = L.config()
    model = executed_mac_model(cfg, nbits)
    peak_gmac, how = measured_int_peak(local)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except Exception:
        pass
    hbm_peak = peaks.get('hbm_gbs', 6650.0)

    def short(k):
        return k.replace('zk::', '')

    def kernel_roofline(pr, name, nsteps, macs_per_item, alg_bytes_per_item, what):
        e = next((v for k, v in pr.items() if short(k) == name), None)
        if not e or not e['launches']:
            return None
        avg_ms = e['ms'] / e['launches']
        per_launch = e['items'] / e['launches']
        ach = e['items'] * macs_per_item / (e['ms'] * 1e-3) / 1e9
        return {'kernel': f'zk_task_kernel<{name}> ({what})',
                'bound': 'int32-multiplier pipe (IMAD.WIDE.U32, fmaheavy) — not hbm/tensor: ~30 modmul per HBM byte',
                'achieved': ach, 'peak': peak_gmac, 'unit': 'G(32x32+64 MAC)/s', 'frac': ach / peak_gmac,
                'peak_source': how, 'mac_count': 'executed (117 IMAD.WIDE per 258-bit product)',
                'avg_launch_ms': avg_ms, 'launches_per_step': e['launches'] / nsteps, 'items_per_launch': per_launch,
                'hbm': {'achieved': per_launch * alg_bytes_per_item / (avg_ms * 1e-3) / 1e9, 'peak': hbm_peak, 'unit': 'GB/s',
                        'frac': per_launch * alg_bytes_per_item / (avg_ms * 1e-3) / 1e9 / hbm_peak,
                        'peak_source': 'MEASURED_PEAKS.json' if peaks else 'fallback 6.65 TB/s'}}

    def whole_step(pr, nsteps, step_ms, extra=None):
        macs = 0.0
        for k, e in pr.items():
            m = (extra or {}).get(short(k), model.get(short(k), 0.0))
            macs += e['items'] * m
        macs /= nsteps
        return {'executed_gmac_per_step': macs / 1e9, 'achieved': macs / (step_ms * 1e-3) / 1e9, 'peak': peak_gmac,
                'frac': macs / (step_ms * 1e-3) / 1e9 / peak_gmac, 'unit': 'G(32x32+64 MAC)/s',
                'note': 'sum over the modelled kernels of items x executed MACs per item (bench.py executed_mac_model; '
                        'unlisted kernels count as zero) / ms_per_step of the timed region / measured peak'}

    roof = kernel_roofline(prof, 'TomCommitHTask', psteps, model['TomCommitHTask'], 32 + 144 + 108,
                           f"fixed-base Pedersen commitments C = K + r*h, 258-bit field, a=-1 image curve: {cfg['tom_nwin']} "
                           'lookups x 7 modmul x 117 MAC per item')
    if roof:
        ms_c = sum(e['ms'] for k, e in prof.items() if short(k) in ('TomCommitHTask', 'TomCommitGTask', 'TomCommitTask'))
        mac_c = sum(e['items'] * model[short(k)] for k, e in prof.items() if short(k) in ('TomCommitHTask', 'TomCommitGTask', 'TomCommitTask'))
        roof['share_of_step'] = next(e['ms'] for k, e in prof.items() if short(k) == 'TomCommitHTask') / (ms_prof_step * psteps)
        roof['all_commit_kernels'] = {'share_of_step': ms_c / (ms_prof_step * psteps), 'achieved': mac_c / (ms_c * 1e-3) / 1e9,
                                      'frac': mac_c / (ms_c * 1e-3) / 1e9 / peak_gmac}
        roof['whole_step'] = whole_step(prof, psteps, ms_step)
        per_lookup = NCU_DRAM_BYTES_PER_LOOKUP.get(cfg['tom_w'])
        roof['traffic'] = roof['items_per_launch'] * (284.0 + per_lookup * cfg['tom_nwin']) if per_lookup else None
        roof['traffic_unit'] = 'bytes/launch'
        roof['traffic_note'] = ('algorithmic bytes are 284 B/commitment; the rest is the random 128-byte table lookups '
                                f"({cfg['tom_nwin'] * ((1 << (cfg['tom_w'] - 1)) + 1) * 128 / 1e6:.0f} MB signed-digit table per base, ncu capture in profiles/) — HBM stays < 15 % busy")
    # verifier: the Pippenger window kernel (one thread per (proof, window); multiW + GK instances in one grid)
    ent_w = 2 + 20 * (2 + 32 * zero_bits / 80.0)      # expected variable points of multiW for this batch
    ent_g = 4 * nbits + 1
    msm_macs = ((ent_w + ent_g) * 63 / 64 * 8 + 2 * 64 * 9) * MAC_PER_TOM_MODMUL      # per (proof, window): both instances
    vextra = {'MsmTomWindowBothTask': msm_macs / 2,       # items counts both instances' threads
              'MsmCombineAllTask': ((258 * 8 + 43 * 9) * 2 * MAC_PER_TOM_MODMUL + (256 * 13 + 64 * 14) * MAC_PER_P256_MODMUL) / 3,
              'VValidateTask': (2 + 32 * zero_bits / 80.0) * 7 * MAC_PER_TOM_MODMUL}
    agg_c = agg_c_prof
    agg_name = 'AggBucketTask<AggTomSrc>'
    agg_e = next((v for k, v in vprof.items() if short(k) == agg_name), None)
    agg_on = bool(agg_e and agg_e['ms'] > 0 and agg_c > 0)
    if agg_on:
        # chunk-wide aggregate check: ONE wide-window MSM per chunk, one thread per (window, bucket); every entry costs
        # one mixed addition (8 modmul) in every window; the bucket tree costs ~2.1 additions (9 modmul) per bucket
        nwin = -(-258 // agg_c)
        entries = B * (ent_w + ent_g)
        vextra['AggBucketTask<AggTomSrc>'] = entries * nwin * 8 * MAC_PER_TOM_MODMUL / (agg_e['items'] / 2)
        lv = next((v for k, v in vprof.items() if short(k) == 'AggLevelTask<AggTomSrc>'), None)
        if lv and lv['items']:
            vextra['AggLevelTask<AggTomSrc>'] = (agg_e['items'] / 2) * 2.1 * 9 * MAC_PER_TOM_MODMUL / (lv['items'] / 2)
        vroof = kernel_roofline(vprof, agg_name, 2, vextra[agg_name], (128 + 4 + 32 / nwin) * entries * nwin / (agg_e['items'] / 2) + 144,
                                f'aggregate check of a whole chunk: signed {agg_c}-bit windows x {nwin}, ~{ent_w + ent_g:.0f} points per '
                                'proof, one thread per (window, bucket), 8 modmul per bucket addition x 117 MAC')
    else:
        vroof = kernel_roofline(vprof, 'MsmTomWindowBothTask', 2, msm_macs / 2, (ent_w + ent_g) / 2 * (128 + 32) / 43 + 144,
                                f'sorted-bucket Pippenger, signed 6-bit windows: ~{ent_w:.0f} + {ent_g} points per proof, '
                                '8 modmul per bucket addition + 2 x 32 x 9 for the running sums, x 117 MAC')
    if vroof and agg_on:
        vroof['traffic'] = entries * nwin * NCU_DRAM_BYTES_PER_AGG_ENTRY_WINDOW / vroof['launches_per_step']
        vroof['traffic_unit'] = 'bytes/launch'
        vroof['traffic_note'] = ('scaled from the ncu capture in profiles/pipes_r2m_config2.md; algorithmic: 132 B per (entry, window) — '
                                 'L2 serves a fifth of the entry reads')
    if vroof:
        vroof['share_of_step'] = next(e['ms'] for k, e in vprof.items() if short(k) == (agg_name if agg_on else 'MsmTomWindowBothTask')) / (ms_vprof_step * 2)
        if agg_on:
            for k in ('MsmTomWindowBothTask', 'MsmCombineAllTask'):      # they return at once after an accepted aggregate
                vextra[k] = 0.0
        vroof['whole_step'] = whole_step(vprof, 2, v_ms, vextra)
        vroof['aggregate'] = {'window_bits': agg_c, 'chunks_accepted': L.stat('agg_pass'), 'chunks_per_proof_path': L.stat('agg_fail'),
                              'note': 'zk_verify_agg.cuh: the sum over all proofs of a chunk of the three linear combinations '
                                      '(every relation has its own random scalar, multimult.ts:147-174) is checked first; the '
                                      'per-proof MSMs run only for a chunk whose sum is not the identity (ZKA_AGG=0: always)'} if agg_on else None

    def kern(pr, nsteps):
        return {short(k): {'ms_per_step': round(v['ms'] / nsteps, 4), 'launches_per_step': v['launches'] / nsteps}
                for k, v in sorted(pr.items(), key=lambda kv: -kv[1]['ms'])}
    cpu = cpu_baseline(N) if world == 1 and not args.no_cpu else None
    line = {
        'metric': 'ZKAttest proofs/sec', 'value': value, 'unit': 'proofs/s', 'n_gpus': world,
        'steps': args.steps, 'warmup': max(args.warmup, 3), 'ms_per_step': ms_step, 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': 'u256/u258 (32-bit limbs, Montgomery)', 'data': 'synthetic',
        'config': {'workload': f'{wname}: batch {B} proofs per GPU, ring N={N}, SecLevel {SEC_LEVEL}, '
                               f'P-256 + tomEdwards256 (BASELINE.json configs[{ {"config1": 1, "config2": 2, "config3": 3}.get(wname, "-") }]'
                               + ('; verify leg = configs[4])' if wname == 'config3' else ')'),
                   'l2': 'working set per step > L2 (tape + proofs ~2.6 GB at 8192 proofs) and a 256 MiB buffer is rewritten between steps',
                   'tom_window_bits': cfg['tom_w'], 'chunk': cfg['chunk'], 'lanes': cfg.get('lanes'),
                   'collective': 'none' if world == 1 else {
                       'pipeline': "the NCCL all-gather of step k's proof bytes overlaps the proving of step k + 1 (two output "
                                   'buffer sets); the timed K steps end when the last gather has landed; ',
                       'serial': "the NCCL all-gather of a step's proof bytes follows the step (exposed); ",
                       'chunks': 'one prove call per step, finished chunks are gathered while later ones are proved; ',
                       'groups': 'sub-batches proved by separate calls, a finished one is gathered while the next is proved; ',
                   }[mode] + gather.describe()},
        'e2e': {'value': world * B / (e2e_ms * 1e-3), 'unit': 'proofs/s', 'h2d_bytes_per_step': h2d,
                'd2h_bytes_per_step': d2h, 'ms_per_step': e2e_ms, 'bit_identical_to_device_arm': same,
                'tape_generation': {'s_per_proof': tape_gen_s_per_proof, 'bytes_per_proof': ts,
                                    'note': 'os.urandom + rnd() rejection (api.synth_os_tape), one host thread; NOT inside the timed '
                                            'region — the C ABI takes the randomness tape as an input buffer'}},
        'gpu_launches': launches,
        'clocks': clocks,
        'roofline': roof,
        'cpu_baseline': cpu,
        'ref_equiv_modmul_per_s': value * W_PROVE_REF.get(N, 6.9e6),
        'verify': {'metric': 'ZKAttest verifies/sec', 'value': world * B / (v_ms * 1e-3), 'unit': 'verifies/s', 'ms_per_step': v_ms,
                   'all_accepted': all_ok, 'gpu_launches_per_step': vlaunches,
                   'collective': 'none' if world == 1 else 'one NCCL all-gather of ok[] (1 byte per proof) per step',
                   'e2e': {'value': world * B / (ve2e_ms * 1e-3), 'unit': 'verifies/s', 'ms_per_step': ve2e_ms,
                           'h2d_bytes_per_step': v_h2d, 'd2h_bytes_per_step': 5 * B, 'all_accepted': v_e2e_ok,
                           'note': 'host proofs, messages, ring and verifier tape in; ok[] and status[] out'},
                   'note': 'zka_verify_batch over the proofs of the last prove step, secparam 20 (zkpAttestList.ts:177)',
                   'roofline': vroof, 'kernels': kern(vprof, 2)},
        'kernels': kern(prof, psteps),
        'kernels_note': 'per-kernel CUDA-event pairs from a separate un-timed pass on ONE lane (sum '
                        f'{ms_prof_step:.2f} ms/step prove, {ms_vprof_step:.2f} ms/step verify; the timed steps run `lanes` lanes concurrently)',
    }
    if gather_info:
        line['gather'] = gather_info
    emit_json(line)
    if world > 1:
        dist.destroy_process_group()


_REAL_STDOUT = None


def quiet_stdout():
    """Route fd 1 to stderr while the run is in progress: NCCL (version banner) and other native
    libraries write to stdout, but the contract is ONE JSON line there."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit_json(line):
    sys.stdout.flush()
    data = (json.dumps(line) + '\n').encode()
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, data)


def main():
    quiet_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--workload', default=None, choices=sorted(WORKLOADS),
                    help='default: config2 on one GPU, config3 (8192 per GPU x ring 1024) under torchrun')
    ap.add_argument('--gather-mode', default='pipeline', choices=['pipeline', 'serial', 'chunks', 'groups'],
                    help='N>1: how the all-gather of the proof bytes overlaps proving (see run_ours)')
    ap.add_argument('--gather-groups', type=int, default=2, help='N>1, --gather-mode groups: sub-batches per step')
    ap.add_argument('--gather-chunk', type=int, default=1408,
                    help='N>1, --gather-mode chunks: largest chunk of the prove call (two chunks per lane at 8192 proofs, 3 lanes)')
    ap.add_argument('--batch', type=int, default=0)
    ap.add_argument('--ring', type=int, default=0)
    ap.add_argument('--no-cpu', action='store_true', help='skip the cpu_baseline leg')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='after the timed steps, write what the last one returned to DIR/<name>.npy (float32): proofs '
                         '(a seeded sample of rows when all of them exceed 60 MiB; proof_rows names them), proof_len, '
                         'status and, for --impl ours, verify_ok / verify_status of the timed verify leg; rank 0 only')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_ours(args)


if __name__ == '__main__':
    main()
