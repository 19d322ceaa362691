"""The attention kernels against a float64 restatement of BertSelfAttention (M.py:241-256) across every sequence-length class
and with many work items per CTA.

The default kernels are persistent: `min(B*A, SMs)` CTAs each walk the items blockIdx.x + li * gridDim.x, and the TMA /
mbarrier ring stage (li % 2), its wait parity ((li / 2) & 1) and the row offset of the short second tile (li & 3) all depend
on the CTA-local index li. So every persistent case is sized to B*A >= 5 * SMs with B*A % SMs != 0: each CTA reaches li >= 4
(both ring stages wrap, every row offset occurs) and the CTAs finish unevenly.

The sequence lengths sit on both sides of each dispatch switch of vb_attention.cu (forward / backward):
  S 1-128    tcgen05, one query tile          / tcgen05, one key tile, 2-stage ring
  S 129-176  tcgen05, two query tiles         / tcgen05, two key tiles, 2-stage ring
  S 177-192  tcgen05, two query tiles         / tcgen05, two key tiles, 1-stage ring (2 stages exceed 227 KB)
  S 193-256  whole-head mma.sync (13-16 warps) / whole-head mma.sync
  S > 256    staged                            / staged
The masks follow the production layout [text | text padding | regions | region padding], and a few examples in the middle
and at the end of the batch are fully masked. Outputs live in NaN-filled slices of larger buffers: a row that is never
written fails the finiteness check, and a write past the end changes the guard tail.

test_forced_implementation reruns the file with the alternative kernels forced (the switches are read once per process).
"""
import ctypes
import os
import random

import pytest
import torch

pytestmark = pytest.mark.gpu

SEQ_LENS = [1, 17, 64, 65, 76, 128, 129, 136, 164, 176, 177, 185, 192, 193, 240, 256, 257, 356]
A = 12                    # production head count
P_DROP = 0.1
N_DROP = 26               # p = 0.1 quantised to n / 256 (DESIGN.md §2)
DROP_SCALE = 256.0 / (256.0 - N_DROP)
GUARD_ROWS = 256          # guard tail after each output, in rows of that output


def _staged_forced():
    return os.environ.get("VB_ATTN_STAGED", "0") not in ("", "0")


def _head_forced():
    return os.environ.get("VB_ATTN_FWD_IMPL", "").startswith("h")


def _batch(S, sms):
    """B for A = 12 heads: the smallest with B*A >= 5 * SMs and B*A not a multiple of SMs (the staged kernels above S = 256
    are not persistent, so a small batch is enough there)."""
    if S > 256:
        return 6
    B = -(-5 * sms // A)
    while (B * A) % sms == 0:
        B += 1
    return B


def _production_bias(B, S, seed):
    """additive mask bias [B, S]: per example valid text, text padding, valid regions, region padding (random lengths),
    and fully masked examples (-10000 everywhere: uniform attention over the raw scores, M.py:1293) spread over the batch."""
    rng = random.Random(seed)
    bias = torch.full((B, S), -10000.0)
    fully = sorted({B // 3, (2 * B) // 3, B - 1})
    for b in range(B):
        if b in fully:
            continue
        T = rng.randint(1, S)           # text segment (the regions take the rest)
        bias[b, :rng.randint(1, T)] = 0.0
        bias[b, T:T + rng.randint(0, S - T)] = 0.0
    return bias, fully


def _guarded(rows, cols, dtype, dev):
    """NaN-filled [rows, cols] view at the start of a buffer with GUARD_ROWS more rows; returns (view, buffer)."""
    buf = torch.full(((rows + GUARD_ROWS) * cols,), float("nan"), device=dev, dtype=dtype)
    return buf[:rows * cols].view(rows, cols), buf


def _tail_bits(buf, n):
    t = buf[n:]
    return t.view(torch.int16 if t.dtype == torch.bfloat16 else torch.int32).clone()


def _rel(out, ref):
    out, ref = out.double(), ref.double()
    assert torch.isfinite(out).all()
    return ((out - ref).abs().max() / ref.abs().max().clamp_min(1e-9)).item()


def _reference(qkv, bias, B, S, keep=None):
    """M.py:241-256 in float64 on the bf16 inputs: scale 1/8, additive bias, softmax, dropout on the probabilities, P V,
    heads merged. Returns (leaf qkv, ctx [B*S, H], lse [B, A, S])."""
    x = qkv.double().requires_grad_(True)
    q, k, v = x.view(B, S, 3, A, 64).permute(2, 0, 3, 1, 4)
    sc = q @ k.transpose(-1, -2) / 8.0 + bias.double()[:, None, None, :]
    p = torch.softmax(sc, -1)
    if keep is not None:
        p = p * keep * DROP_SCALE
    return x, (p @ v).permute(0, 2, 1, 3).reshape(B * S, A * 64), torch.logsumexp(sc, -1)


def _unpack(words, n, nkb):
    """[n, nkb*64, nkb] 64-bit words -> [n, nkb*64, nkb*64] bool (bit j of word w = column 64 w + j)."""
    return ((words.unsqueeze(-1) >> torch.arange(64, device=words.device)) & 1).bool().reshape(n, nkb * 64, nkb * 64)


@pytest.mark.parametrize("p_drop", [0.0, P_DROP], ids=["nodrop", "drop"])
@pytest.mark.parametrize("S", SEQ_LENS, ids=[f"S{s}" for s in SEQ_LENS])
def test_attention_matches_float64_reference(S, p_drop):
    from visualbert_b200 import _lib
    staged = _staged_forced() or S > 256
    if _head_forced() and S > 256:
        pytest.skip("the whole-head kernels cover S <= 256")
    L = _lib.lib()
    dev = torch.device("cuda:0")
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    B = _batch(S, sms)
    items = B * A
    if not staged:   # persistent kernels: every CTA gets >= 5 items, and not all the same number
        assert items >= 5 * sms and items % sms != 0, (items, sms)
    H = A * 64
    torch.manual_seed(1000 + S)
    qkv = torch.randn(B * S, 3 * H, device=dev).bfloat16()
    dctx = torch.randn(B * S, H, device=dev).bfloat16()
    bias, fully = _production_bias(B, S, seed=S)
    bias = bias.to(dev)

    ctx, ctx_buf = _guarded(B * S, H, torch.bfloat16, dev)
    lse, lse_buf = _guarded(items, S, torch.float32, dev)
    dqkv, dqkv_buf = _guarded(B * S, 3 * H, torch.bfloat16, dev)
    drow, drow_buf = _guarded(items, S, torch.float32, dev)
    tails = [(b, t.numel(), _tail_bits(b, t.numel())) for t, b in ((ctx, ctx_buf), (lse, lse_buf), (dqkv, dqkv_buf), (drow, drow_buf))]
    nkb = (S + 63) // 64
    keep = torch.zeros(int(L.vb_attention_keep_bytes(B, S, A)), device=dev, dtype=torch.uint8) if p_drop else None
    P = lambda t: ctypes.c_void_p(t.data_ptr()) if t is not None else None
    drop = (ctypes.c_float(p_drop), ctypes.c_uint64(0x5EED0000 + S), 7, st)
    _lib.check(L.vb_attention_fwd(P(qkv), P(bias), P(ctx), P(lse), P(keep), B, S, A, H, *drop), "attn_fwd")
    _lib.check(L.vb_attention_bwd(P(qkv), P(bias), P(ctx), P(lse), P(keep), P(dctx), P(dqkv), P(drow), B, S, A, H, *drop),
               "attn_bwd")
    torch.cuda.synchronize()

    for buf, n, before in tails:   # nothing written past the end of any output
        assert torch.equal(_tail_bits(buf, n), before)

    keep_ref = None
    if p_drop:
        both = keep.view(torch.int64).view(2, items, nkb * 64, nkb)   # [0]: rows = queries, [1]: the transpose (rows = keys)
        bits = _unpack(both[0], items, nkb)[:, :S, :S]
        if not staged:   # the staged kernels draw their own bits, query-major only
            assert torch.equal(bits, _unpack(both[1], items, nkb)[:, :S, :S].transpose(1, 2))
        q = N_DROP / 256.0
        frac = bits.float().mean().item()
        assert abs(frac - (1 - q)) < 6 * (q * (1 - q) / bits.numel()) ** 0.5 + 1e-4, frac
        if S * S >= 64:   # every (b, h) item draws its own mask (a mask indexed by li would repeat across items)
            w = torch.rand(S * S, device=dev, dtype=torch.float64, generator=torch.Generator(device=dev).manual_seed(S))
            assert torch.unique(bits.reshape(items, S * S).double() @ w).numel() == items
        keep_ref = bits.view(B, A, S, S).double()

    x, ref, lse_ref = _reference(qkv, bias, B, S, keep_ref)
    err = {"ctx": _rel(ctx, ref)}
    assert torch.isfinite(lse).all()
    err["lse"] = (lse.view(B, A, S).double() - lse_ref).abs().max().item()
    ref.backward(dctx.double())
    for i, name in enumerate(("dq", "dk", "dv")):
        if S == 1 and name != "dv":
            # one key: the softmax is 1 and the exact dQ, dK are zero. The kernels' dS = P (dP - D) is then the residue of
            # D = rowsum(dO * O) taken over the bf16 O (measured 1e-6 without dropout, 2e-2 with), so dQ = dS K / 8 and
            # dK = dS Q / 8 are bounded by that residue instead of by a relative error
            resid = (dctx.double() * (ctx.double() - ref.detach())).view(B, A, 64).sum(-1).abs().max().item()
            other = qkv[:, (1 - i) * H:(2 - i) * H].double().abs().max().item()
            got = dqkv[:, i * H:(i + 1) * H].double()
            assert torch.isfinite(got).all()
            err[name + "_abs"] = got.abs().max().item()
            assert err[name + "_abs"] <= 1.5 * resid * other / 8.0 + 1e-4, (err, resid)
            continue
        err[name] = _rel(dqkv[:, i * H:(i + 1) * H], x.grad[:, i * H:(i + 1) * H])
    # D = rowsum(dO * O) over the kernel's own O, as the backward uses it
    d_ref = (dctx.double() * ctx.double()).view(B, S, A, 64).sum(-1).permute(0, 2, 1)
    assert torch.isfinite(drow).all()
    err["drow"] = (drow.view(B, A, S).double() - d_ref).abs().max().item() / d_ref.abs().max().item()
    print(f"S={S} B={B} p={p_drop} fully_masked={fully} errors: " + " ".join(f"{k}={v:.2e}" for k, v in err.items()))
    assert err["ctx"] < 1e-2, err
    assert err["lse"] < 2e-2, err
    for name in ("dq", "dk", "dv"):
        assert err.get(name, 0.0) < 2e-2, err
    assert err["drow"] < 2e-3, err


FORCED = {
    "head": {"VB_ATTN_FWD_IMPL": "head", "VB_ATTN_BWD_IMPL": "head"},             # S <= 176 reaches the P/dS-in-shared backward
    "head_nops": {"VB_ATTN_FWD_IMPL": "head", "VB_ATTN_BWD_IMPL": "head", "VB_ATTN_BWD_PS": "0"},
    "staged": {"VB_ATTN_STAGED": "1"},
}


@pytest.mark.parametrize("impl", list(FORCED), ids=list(FORCED))
def test_forced_implementation(impl):
    """The sweep again with the whole-head kernels (with and without the P/dS-in-shared backward) or the staged kernels
    forced; the switches are read once per process, so each runs in a subprocess."""
    import subprocess, sys
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-m", "gpu", "-q", "-k", "not forced_implementation"],
                       env=dict(os.environ, **FORCED[impl]), capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
