"""BASELINE config 5: 3D grounding, N=200k points x P=256 prompts x C=768 (fp16 and fp32 features).
Prints one JSON line per case with CUDA-event timings of the GEMM+epilogue and of the whole predict()."""
import json, os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from dropclip_b200 import _lib
from dropclip_b200.engine import FusionEngine

def ev():
    return torch.cuda.Event(enable_timing=True)

def main():
    n, p, c = 200_000, 256, 768
    eng = FusionEngine("cuda")
    g = torch.Generator(device="cuda").manual_seed(0)
    peaks = json.load(open(os.path.join(os.path.dirname(__file__), "..", "MEASURED_PEAKS.json"))) if os.path.exists(
        os.path.join(os.path.dirname(__file__), "..", "MEASURED_PEAKS.json")) else {}
    for dtype in (torch.float16, torch.float32):
        x0 = torch.randn((n, c), generator=g, device="cuda").to(dtype)
        t = torch.randn((p, c), generator=g, device="cuda")
        t = (t / t.norm(dim=-1, keepdim=True)).to(dtype)
        flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
        for mode, name in ((_lib.DC_GROUND_PAIRED, "paired"), (_lib.DC_GROUND_ARGMAX, "argmax"), (_lib.DC_GROUND_RAW, "raw")):
            times = []
            for it in range(8):
                x = x0.clone()
                flush.zero_()
                a, b = ev(), ev()
                a.record()
                if mode != _lib.DC_GROUND_RAW:
                    out, pred = eng.predict(x, t, mode, 0.1, True, 0.7)  # one library call (dc_predict)
                else:
                    out, pred, mm = eng.ground(x, t, mode, 0.1, normalize=True)
                b.record()
                torch.cuda.synchronize()
                if it >= 3:
                    times.append(a.elapsed_time(b))
            ms = sorted(times)[len(times) // 2]
            terms = 1 if dtype == torch.float16 else 3
            flops = 2.0 * n * c * p
            es = 2 if dtype == torch.float16 else 4
            alg_bytes = n * c * es * 2 + p * c * es + n * 5 + (n * p * 4 if name == "raw" else 0)  # read + in-place write-back
            print(json.dumps({"case": f"ground_{name}_{'f16' if dtype == torch.float16 else 'f32'}", "ms": ms,
                              "points_per_s": n / (ms * 1e-3), "useful_tflops": flops / (ms * 1e-3) / 1e12,
                              "issued_tflops": flops * terms / (ms * 1e-3) / 1e12, "alg_GBps": alg_bytes / (ms * 1e-3) / 1e9,
                              "frac_hbm": alg_bytes / (ms * 1e-3) / 1e9 / peaks.get("hbm_gbs", 6650.0),
                              "frac_tensor_useful": flops / (ms * 1e-3) / 1e12 / peaks.get("bf16_tflops", 1590.0)}))

if __name__ == "__main__":
    main()
