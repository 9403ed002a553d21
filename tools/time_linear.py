"""Cross-encoder linear layer as rl_xenc_linear dispatches it (weight-resident kernel for K <= 384, streaming
kernel otherwise): parity of every GEMM shape against torch (incl. a ragged token count), then CUDA-event timing
of back-to-back launches.  ``--bert-base`` times the BERT-base shapes (hidden 768, FFN 3072: ms-marco-MultiBERT-L-12)
instead of the MiniLM ones."""
import argparse
import json
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
from raglite_b200 import _lib  # noqa: E402

lib = _lib.load()
g = torch.Generator().manual_seed(0)
T = 51200 + 77   # ragged: the last token tile is partial
ap = argparse.ArgumentParser()
ap.add_argument("--bert-base", action="store_true")
args = ap.parse_args()
shapes = [("qkv", 1152, 384, 0), ("out", 384, 384, 0), ("ffn_up", 1536, 384, 1), ("ffn_down", 384, 1536, 0)]
if args.bert_base:
    shapes = [("qkv", 2304, 768, 0), ("out", 768, 768, 0), ("ffn_up", 3072, 768, 1), ("ffn_down", 768, 3072, 0)]
out = {}
s = torch.cuda.current_stream().cuda_stream
for name, N, K, act in shapes:
    X = (torch.randn((T, K), generator=g) * 0.5).half().cuda()
    W = (torch.randn((N, K), generator=g) / K**0.5).float().cuda()
    b = torch.randn(N, generator=g).float().cuda()
    img = torch.empty(lib.rl_xenc_linear_image_bytes(N, K), dtype=torch.uint8, device="cuda")
    assert lib.rl_xenc_pack_linear(W.data_ptr(), N, K, img.data_ptr(), s) == 0
    ref = X[:4096].float() @ W.half().float().T + b
    if act:
        ref = torch.nn.functional.gelu(ref)
    Y = torch.empty((T, N), dtype=torch.float16, device="cuda")
    Y.zero_()
    assert lib.rl_xenc_linear(X.data_ptr(), img.data_ptr(), b.data_ptr(), Y.data_ptr(), T, N, K, act, s) == 0, lib.rl_last_error()
    torch.cuda.synchronize()
    err = (Y[:4096].float() - ref).abs().max().item()
    tail_err = (Y[-128:].float() - (torch.nn.functional.gelu(X[-128:].float() @ W.half().float().T + b) if act
                                    else X[-128:].float() @ W.half().float().T + b)).abs().max().item()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(3):
        lib.rl_xenc_linear(X.data_ptr(), img.data_ptr(), b.data_ptr(), Y.data_ptr(), T, N, K, act, s)
    e0.record()
    for _ in range(20):
        lib.rl_xenc_linear(X.data_ptr(), img.data_ptr(), b.data_ptr(), Y.data_ptr(), T, N, K, act, s)
    e1.record()
    torch.cuda.synchronize()
    us = e0.elapsed_time(e1) / 20 * 1e3
    out[name] = {"us": round(us, 1), "tflops": round(2.0 * T * N * K / us / 1e6, 1), "max_err": err, "tail_err": tail_err}
print(json.dumps(out))
