"""Cost of the float64 re-evaluation path: C3 2^20 fp32, graph replay over 6 batches, with the study knob
H2O_NO_FALLBACK = 1 (never) / k (exactly every k-th body) / 0 (the real flags)."""
import os, subprocess, sys, json
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for k in os.environ.get("KS", "1,0,1048576,65536,8192,1024,128,16,1").split(","):
    if k == "1" and "done1" in globals():
        k_env = "2"  # k = 1 means "never"; every body = every 2nd... use a dedicated value below
    env = dict(os.environ, H2O_NO_FALLBACK=k)
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1200", "--warmup", "5", "--no-cpu-baseline",
                          "--no-extra", "--no-e2e", "--regions", "60"], env=env, capture_output=True, text=True)
    d = json.loads(res.stdout.strip().splitlines()[-1])
    t = d["extra"]["timing"]
    print(f"H2O_NO_FALLBACK={k:>8s}: median {1e3 * t['ms_per_step_median']:.2f} us  p10 {1e3 * t['ms_per_step_p10']:.2f}  "
          f"re-evaluated {int(d['global_stats']['reevaluated_bodies'])}  clk {d['clocks']['sm_mhz']}", flush=True)
    done1 = True
