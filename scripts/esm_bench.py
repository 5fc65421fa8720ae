"""ESM-2 receptor embeddings (``esm.ESM2`` / ``esm.embed_sequences``) on one GPU: a random-init 33-layer, 1280-wide model
(the 650M shape) on single chains of 150, 300, 600 and 1022 residues and on one protein of four chains (one
``embed_sequences`` call, one padded batch).

Timing: CUDA events over windows of at least 1 s after warm-up, median of the repeats.  Per protein: milliseconds per
call, the summed time of its ``ddp_esm_attention`` launches (CUDA events around each launch, in separate windows), the
attention's FLOP/s against the FP32 data-sheet rate, and the whole forward's FLOP/s computed from shapes (GEMMs +
attention, 2 FLOPs per multiply-add).  Comparison line: the same forward in plain PyTorch fp32 ops on the same device
(``oracle/esm2_ref.py`` run in fp32: materialised [T, T] scores, torch softmax / layer norm / erf).  The card's name
and power limit are read in the same run.  Writes ``profiles/esm_bench.json``.

    python scripts/esm_bench.py [--repeats 5] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from diffdock_pocket_b200 import esm  # noqa: E402
from oracle import esm2_ref  # noqa: E402

# NVIDIA B200 FP32 (CUDA cores), dense: the HGX B200 data sheet's 600 TFLOP/s for eight GPUs, per GPU.  The data sheet
# assumes a card allowed up to 1000 W; the power limit read below is recorded beside every rate.
FP32_DATASHEET_TFLOPS = 75.0
PROTEINS = [('L150', [150]), ('L300', [300]), ('L600', [600]), ('L1022', [1022]), ('4chains', [310, 262, 198, 145])]


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = 'unknown'
    return name, q


def flops(lengths, T, D=1280, H=20, layers=33):
    """(whole forward, attention) FLOPs of one padded batch: GEMMs over every B x T row (Q/K/V, out_proj, fc1, fc2 =
    24 N D^2 per layer) and the attention as the kernel computes it (every query row of T against the L_b keys: 4 T L_b D)."""
    N = len(lengths) * T
    att = layers * sum(4 * T * L * D for L in lengths)
    return layers * 24 * N * D * D + att, att


def timed(fn, repeats):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def window(n):
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / 1e3

    window(2)                                             # warm-up: module load, library algorithm choice
    iters = max(1, int(np.ceil(1.1 / max(window(2) / 2, 1e-6))))
    per = []
    while len(per) < repeats:
        t = window(iters)
        if t < 1.0:                                       # every timed window lasts at least 1 s
            iters = int(np.ceil(iters * 1.1 / t))
            continue
        per.append(t / iters)
    return float(np.median(per)), per


def attention_time(model, tokens, lengths, repeats):
    """Summed seconds of the ddp_esm_attention launches of one forward (events around each launch)."""
    orig = esm.attention
    events = []

    def wrapped(*a):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        orig(*a)
        e.record()
        events.append((s, e))

    esm.attention = wrapped
    try:
        sums = []
        for _ in range(repeats):
            events.clear()
            model(tokens, lengths)
            torch.cuda.synchronize()
            sums.append(sum(s.elapsed_time(e) for s, e in events) / 1e3)
    finally:
        esm.attention = orig
    return float(np.median(sums))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--repeats', type=int, default=5)
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'esm_bench.json'))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit('esm_bench: no CUDA device (every number would be "not measured")')
    dev = torch.device('cuda:0')
    name, limits = card()
    torch.manual_seed(0)
    model = esm.ESM2(33, 1280, 20).to(dev)
    sd = model.state_dict()
    rng = np.random.RandomState(0)
    rows = []
    for tag, chains in PROTEINS:
        seqs = [''.join(rng.choice(list('ACDEFGHIKLMNPQRSTVWY'), n)) for n in chains]
        tokens, lengths = esm.Alphabet().encode(seqs)
        T = tokens.shape[1]
        t_call, reps = timed(lambda: esm.embed_sequences(model, seqs), a.repeats)
        t_att = attention_time(model, tokens, lengths, a.repeats)
        tok_d = tokens.to(dev)
        t_torch, _ = timed(lambda: esm2_ref.forward(sd, tok_d, 33, 20, dtype=torch.float32), a.repeats)
        f_all, f_att = flops(lengths, T)
        with torch.no_grad():
            got = model(tokens, lengths)
            ref = esm2_ref.forward(sd, tok_d, 33, 20, dtype=torch.float32)
        rows.append(dict(
            protein=tag, chains=chains, tokens_per_sequence=T, batch=len(chains),
            ms_per_protein=t_call * 1e3, repeats_ms=[r * 1e3 for r in reps],
            attention_ms=t_att * 1e3, attention_share=t_att / t_call,
            attention_tflops=f_att / t_att / 1e12, attention_of_fp32_datasheet=f_att / t_att / 1e12 / FP32_DATASHEET_TFLOPS,
            forward_tflops=f_all / t_call / 1e12, forward_flops=f_all, attention_flops=f_att,
            plain_torch_fp32_ms=t_torch * 1e3, speedup_vs_plain_torch=t_torch / t_call,
            max_abs_diff_vs_plain_torch=float((got - ref).abs().max()), ref_max_abs=float(ref.abs().max())))
        print(json.dumps(rows[-1]), flush=True)
    out = dict(card=name, power_limit_and_max_sm_clock=limits, torch=torch.__version__,
               fp32_datasheet_tflops=FP32_DATASHEET_TFLOPS, model='random-init ESM2(33, 1280, 20)',
               timing='CUDA events, windows >= 1 s after warm-up, median of repeats; attention_ms = summed events around '
                      'each ddp_esm_attention launch of one forward (separate runs)', proteins=rows)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, 'w') as f:
        json.dump(out, f, indent=1)
    print(json.dumps(dict(card=name, limits=limits)))


if __name__ == '__main__':
    main()
