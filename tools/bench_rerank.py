"""Cross-encoder throughput (BASELINE configs[4]: 1024 queries x 100 candidates) on one GPU, next to the float32
transformers forward on the host cores for a bounded sample and the float16 transformers forward (padded batches,
SDPA attention) on the same GPU and pairs.

  --model minilm     ms-marco-MiniLM-L-12-v2's geometry (H 384, FFN 1536, one label; the default)
  --model multibert  ms-marco-MultiBERT-L-12's geometry (BERT-base: H 768, 12 heads of 64, FFN 3072, two labels)
  --profile CSV      instead of timing: one forward under torch.profiler, per-kernel launch list written to CSV
"""
import argparse, csv, json, subprocess, sys, time
from pathlib import Path
ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT)); sys.path.insert(0, str(ROOT / "tests"))
import numpy as np, torch

ap = argparse.ArgumentParser()
ap.add_argument("--model", choices=("minilm", "multibert"), default="minilm")
ap.add_argument("--pairs", type=int, default=8192)
ap.add_argument("--mean-len", type=int, default=200)
ap.add_argument("--cpu-pairs", type=int, default=64)
ap.add_argument("--tokens-per-call", type=int, default=1 << 18)
ap.add_argument("--hf-batch", type=int, default=64, help="pairs per padded batch of the transformers fp16 arm")
ap.add_argument("--profile", type=Path, default=None)
args = ap.parse_args()

from bert_base_oracle import flashrank_logit_column, seeded_bert_base
from oracle import rerank as orr
from raglite_b200._xenc import CrossEncoderEngine

PEAK_FP16_DENSE = 2250e12   # B200 data sheet, dense fp16, one GPU at 1000 W


def card() -> dict:
    out = {"name": torch.cuda.get_device_name(), "power_limit_w": None, "clocks_max_sm_mhz": None}
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=power.limit,clocks.max.sm",
                            "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=30, check=True)
        p, c = (x.strip() for x in q.stdout.strip().splitlines()[0].split(","))
        out["power_limit_w"], out["clocks_max_sm_mhz"] = float(p), float(c)
    except (OSError, subprocess.SubprocessError, ValueError, IndexError) as e:
        out["query_error"] = repr(e)
    return out


if args.model == "minilm":
    model = orr.seeded_model(seed=0)
    label = "MiniLM-L12-H384"
else:
    model = seeded_bert_base(seed=0)
    label = "MultiBERT-L12 (BERT-base H768)"
cfg = model.config
eng = CrossEncoderEngine.from_hf(model, max_tokens_per_call=args.tokens_per_call)
rng = np.random.default_rng(0)
lens = np.clip(rng.normal(args.mean_len, 60, size=args.pairs).astype(int), 32, 512)
ids = [rng.integers(1000, 30000, size=L).astype(np.int32) for L in lens]
types = [np.r_[np.zeros(12, np.int32), np.ones(L - 12, np.int32)] for L in lens]
eng.score_tokens(ids[:256], types[:256])
torch.cuda.synchronize()

if args.profile is not None:
    # One forward of the whole batch (every packed call), CUDA activity only, summed per kernel name.
    from torch.profiler import ProfilerActivity, profile

    eng.score_tokens(ids, types)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        eng.score_tokens(ids, types)
        torch.cuda.synchronize()
    rows = {a.key: [a.count, a.self_device_time_total] for a in prof.key_averages() if a.self_device_time_total > 0}
    total = sum(v[1] for v in rows.values())
    args.profile.parent.mkdir(parents=True, exist_ok=True)
    with open(args.profile, "w", newline="") as f:
        w = csv.writer(f)
        w.writerow(["kernel", "launches", "total_us", "us_per_launch", "us_per_layer", "share"])
        for name, (n, us) in sorted(rows.items(), key=lambda kv: -kv[1][1]):
            w.writerow([name, n, round(us, 1), round(us / n, 2), round(us / cfg.num_hidden_layers, 1), round(us / total, 4)])
    print(json.dumps({"profile": str(args.profile), "model": args.model, "pairs": args.pairs, "tokens": int(lens.sum()),
                      "device_us_total": round(total, 1), "kernels": len(rows), "card": card()}))
    sys.exit(0)

t0 = time.perf_counter()
logits, scores = eng.score_tokens(ids, types)
torch.cuda.synchronize()
dt = time.perf_counter() - t0
T = int(lens.sum())
H, F, Lyr = cfg.hidden_size, cfg.intermediate_size, cfg.num_hidden_layers
flops = Lyr * (2.0 * T * (3 * H * H + H * H + 2 * H * F) + 4.0 * float((lens.astype(np.float64) ** 2).sum()) * H)

# transformers float16 on the same GPU and pairs: what a user runs without this project (padded batches, SDPA).
from transformers import BertForSequenceClassification

hf = BertForSequenceClassification._from_config(cfg, attn_implementation="sdpa").eval()
hf.load_state_dict(model.state_dict())
hf = hf.half().cuda()
assert hf.config._attn_implementation == "sdpa"


@torch.no_grad()
def hf_fp16(lo: int, hi: int) -> np.ndarray:
    out = []
    for s in range(lo, hi, args.hf_batch):
        chunk_i, chunk_t = ids[s:min(s + args.hf_batch, hi)], types[s:min(s + args.hf_batch, hi)]
        L = max(len(x) for x in chunk_i)
        inp = np.zeros((len(chunk_i), L), np.int64); typ = np.zeros_like(inp); msk = np.zeros_like(inp)
        for r, (a, b) in enumerate(zip(chunk_i, chunk_t)):
            inp[r, :len(a)], typ[r, :len(a)], msk[r, :len(a)] = a, b, 1
        lg = hf(input_ids=torch.from_numpy(inp).cuda(non_blocking=True), token_type_ids=torch.from_numpy(typ).cuda(non_blocking=True),
                attention_mask=torch.from_numpy(msk).cuda(non_blocking=True)).logits
        out.append(lg.float())
    return flashrank_logit_column(torch.cat(out).cpu().numpy())


hf_fp16(0, min(4 * args.hf_batch, args.pairs))
torch.cuda.synchronize()
t0 = time.perf_counter()
hf_logit = hf_fp16(0, args.pairs)
torch.cuda.synchronize()
hf_dt = time.perf_counter() - t0

n = args.cpu_pairs
t0 = time.perf_counter()
ref = flashrank_logit_column(orr.hf_logits(model, ids[:n], types[:n]).reshape(n, -1))
cpu_dt = time.perf_counter() - t0
res = {
    "metric": f"cross-encoder pairs/sec ({label}, packed varlen, fp16 tensor cores)", "pairs": args.pairs,
    "tokens": T, "mean_len": float(lens.mean()), "gpu_pairs_per_s": args.pairs / dt, "gpu_tokens_per_s": T / dt,
    "gpu_tflops": flops / dt / 1e12, "seconds": dt, "c5_seconds_extrapolated": 102400 / (args.pairs / dt),
    "cpu_pairs_per_s": n / cpu_dt, "cpu_threads": torch.get_num_threads(), "cpu_sample_pairs": n,
    "max_abs_logit_err_vs_fp32": float(np.abs(logits[:n] - ref).max()),
}
res.update({
    "model": args.model, "hidden": H, "ffn": F, "layers": Lyr, "heads": cfg.num_attention_heads, "num_labels": cfg.num_labels,
    "flops_per_pass": flops, "share_of_dense_fp16_peak": flops / dt / PEAK_FP16_DENSE,
    "hf_fp16_sdpa_pairs_per_s": args.pairs / hf_dt, "hf_fp16_sdpa_seconds": hf_dt, "hf_batch": args.hf_batch,
    "speedup_vs_hf_fp16": hf_dt / dt, "max_abs_logit_diff_vs_hf_fp16": float(np.abs(logits - hf_logit).max()),
    "card": card(),
})
print(json.dumps(res))
