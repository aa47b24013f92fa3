"""Times decoding from codes at BASELINE configs[1] (B = 32 utterances x 4 s, T' = 320 frames) with CUDA events:
Codec.decode_codes (fac_decode_codes: dequantize + decoder in one call) and model.decoder(outs) (fac_decode on the
dequantized latents) alternately in one run, and fac_dequantize alone (raw C-ABI call, codes validated once up front).
Reports ms per call, audio-seconds per second and the dequantizer's share of the decode call, with the GPU's name, power
limit and SM clock read in the same run.  Prints one JSON line; --out also writes it to a file.

    python scripts/bench_decode_codes.py [--steps 20] [--warmup 3] [--out FILE]

The dequantizer's own inputs and outputs (codes 0.5 MB, outs 42 MB, weights 0.2 MB) fit the 126 MB L2; the decoder's
working set does not.  Timings are therefore of back-to-back calls as an application would make them, not cold-cache.
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader", "-i", "0"], capture_output=True,
                             text=True, timeout=30).stdout.strip()
        return dict(zip(q.split(","), [s.strip() for s in out.split(",")]))
    except Exception as e:             # the numbers are still valid; say that the card could not be read
        return {"error": repr(e)}


def timed(fn, st):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(st)
    fn()
    b.record(st)
    b.synchronize()
    return a.elapsed_time(b)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if a.steps < 12:
        ap.error("--steps must be >= 12")
    if not torch.cuda.is_available():
        sys.exit("needs a CUDA device: nothing is measured on the CPU")
    import facodec_b200 as fb
    from facodec_b200 import synth
    torch.cuda.set_device(0)
    dev = torch.device("cuda:0")
    B, T = 32, 96000
    m = fb.build_model()
    sds = synth.synth_state_dicts(0)
    for k in ("encoder", "quantizer", "decoder"):
        m[k].load_state_dict(sds[k])
        m[k].eval()
    codec = fb.Codec(m)
    x = synth.synth_waves(B, T, seed=2024).to(dev)
    _, codes, timbre = codec.forward(x, n_c=2)
    outs = m.quantizer.from_codes(codes, timbre)[0]
    Tq = codes[0].shape[-1]
    L, h = m.quantizer._engine.L, m.quantizer._engine.handle
    st = torch.cuda.current_stream(dev)
    sp = ctypes.c_void_p(st.cuda_stream)
    o_raw = torch.empty(B, 1024, Tq, device=dev)
    p = lambda t: ctypes.c_void_p(t.data_ptr())

    def dequant():
        rc = L.fac_dequantize(h, p(codes[0]), p(codes[1]), 2, 2, p(codes[2]), 3, 3, p(timbre), B, Tq, p(o_raw), None, None,
                              None, sp)
        assert rc == 0, L.fac_last_error(h)

    calls = {"decode_codes": lambda: codec.decode_codes(codes, timbre), "decoder": lambda: m.decoder(outs),
             "dequantize": dequant}
    for _ in range(a.warmup):
        for fn in calls.values():
            fn()
    torch.cuda.synchronize()
    times = {k: [] for k in calls}
    for _ in range(a.steps):
        for k, fn in calls.items():
            times[k].append(timed(fn, st))
    assert torch.equal(o_raw, outs)
    audio_s = B * Tq * 300 / 24000.0
    res = {"workload": "decode_codes", "config": f"B={B} x 4 s (T'={Tq})", "steps": a.steps, "warmup": a.warmup,
           "gpu": gpu_info()}
    for k, v in times.items():
        med = statistics.median(v)
        res[k] = {"ms_median": round(med, 4), "ms_min": round(min(v), 4), "ms_max": round(max(v), 4),
                  "audio_s_per_s": round(audio_s / (med / 1e3), 1)}
    res["dequantize_share_of_decode_codes"] = round(res["dequantize"]["ms_median"] / res["decode_codes"]["ms_median"], 5)
    res["decode_codes_minus_decoder_ms"] = round(res["decode_codes"]["ms_median"] - res["decoder"]["ms_median"], 4)
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
