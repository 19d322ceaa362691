"""Train-mode (dropout ON) value parity of one BertLayer through the C ABI (vb_layer_fwd / vb_layer_bwd) against the
reference arithmetic (M.py:231-341) in fp32 with THE SAME dropout masks.

The library's dropout is a pure function of (seed, stream, element index) — `dropout_keep8` / `mix32` in
csrc/vb_common.cuh — and the attention-probability bits are written to the keep-mask buffer by the forward. This test
regenerates the hidden-state masks with a torch restatement of that hash, reads the attention bits back, runs the
reference math with those masks and compares the layer output, the input gradient and every parameter gradient.
It covers what eval-mode parity cannot: the forward/backward mask agreement of the tcgen05 attention kernels, the
GEMM-epilogue dropout, and the mask REGENERATION in the LayerNorm backward (dx_drop).
"""
import ctypes
import math

import pytest
import torch

pytestmark = pytest.mark.gpu

M32 = 0xFFFFFFFF


def _mix32(x):
    x = x ^ (x >> 16); x = (x * 0x7feb352d) & M32
    x = x ^ (x >> 15); x = (x * 0x846ca68b) & M32
    return x ^ (x >> 16)


def _mix32_int(x):
    x &= M32
    x ^= x >> 16; x = (x * 0x7feb352d) & M32
    x ^= x >> 15; x = (x * 0x846ca68b) & M32
    return x ^ (x >> 16)


def hidden_keep(seed, stream, rows, cols, p, dev):
    """keep mask [rows, cols] (bool) and survivor scale of vb_common.cuh::dropout_keep8 for a [rows, cols] tensor."""
    n = int(p * 256.0 + 0.5)
    key = _mix32_int((seed & M32) ^ _mix32_int(((seed >> 32) + 0x9E3779B9 * (stream + 1)) & M32))
    idx = torch.arange(rows * cols, device=dev, dtype=torch.int64)
    e8, k = idx >> 3, idx & 7
    kk = key ^ (((e8 >> 31) * 0x27d4eb2f) & M32)
    h = _mix32((((e8 << 1) + (k >> 2)) & M32) ^ kk)
    byte = (h >> (8 * (k & 3))) & 0xFF
    return (byte >= n).view(rows, cols), 256.0 / (256.0 - n)


# The last four rows are BERT-base width (H = 768, A = 12) at B = 64, i.e. 768 attention items: >= 5 per CTA of the persistent
# attention kernels on a 148-SM B200. S = 164 is the benchmark geometry (B*S a multiple of 256: tile-native gelu', fused
# rowsum(dO * O) in the dO GEMM epilogue); S = 185 takes the 1-stage tcgen05 backward, the fused rowsum with an odd sequence
# length and the row-major gelu'; S = 76 a single query tile; S = 200 the whole-head kernels.
@pytest.mark.parametrize("B,S,A,layer_index", [(3, 164, 4, 0), (2, 100, 2, 5), (2, 56, 2, 11),
                                               (64, 164, 12, 3), (64, 185, 12, 7), (64, 76, 12, 1), (64, 200, 12, 9)])
def test_layer_train_mode_matches_reference_math_with_the_same_masks(B, S, A, layer_index):
    from visualbert_b200 import _lib
    L = _lib.lib()
    dev = torch.device("cuda:0")
    if B * A >= 256:   # the production-scale rows: many attention items per CTA, and uneven counts
        sms = torch.cuda.get_device_properties(0).multi_processor_count
        assert B * A >= 5 * sms and B * A % sms != 0, (B * A, sms)
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    torch.manual_seed(17 + layer_index)
    H, I = A * 64, A * 256
    Mr = B * S
    p_h, p_a, seed = 0.1, 0.1, 0x1234567890ABCDEF
    bf = torch.bfloat16
    rnd = lambda *s, sc=1.0: (sc * torch.randn(*s, device=dev))
    x = rnd(Mr, H).to(bf)
    W = dict(qkv=rnd(3 * H, H, sc=0.05).to(bf), o=rnd(H, H, sc=0.05).to(bf), i=rnd(I, H, sc=0.05).to(bf), out=rnd(H, I, sc=0.05).to(bf))
    bvec = dict(qkv=rnd(3 * H, sc=0.1), o=rnd(H, sc=0.1), i=rnd(I, sc=0.1), out=rnd(H, sc=0.1))
    ln = dict(g1=1 + rnd(H, sc=0.1), b1=rnd(H, sc=0.1), g2=1 + rnd(H, sc=0.1), b2=rnd(H, sc=0.1))
    lens = torch.randint(S // 2, S + 1, (B,), device=dev)
    mbias = ((torch.arange(S, device=dev)[None, :] >= lens[:, None]).float() * -10000.0).contiguous()

    # ---- the library: forward + backward through the C ABI ----
    f32 = torch.float32
    e = lambda *s, dt=bf: torch.empty(*s, device=dev, dtype=dt)
    keep = torch.zeros(int(L.vb_attention_keep_bytes(B, S, A)), device=dev, dtype=torch.uint8)
    acts = dict(qkv=e(Mr, 3 * H), ctx=e(Mr, H), lse=e(B, A, S, dt=f32), pre1=e(Mr, H), mean1=e(Mr, dt=f32), rstd1=e(Mr, dt=f32),
                x1=e(Mr, H), u=e(Mr, I), g=e(Mr, I), pre2=e(Mr, H), mean2=e(Mr, dt=f32), rstd2=e(Mr, dt=f32), keep_mask=keep)
    y = e(Mr, H)
    d = _lib.LayerDesc(batch=B, seq=S, hidden=H, heads=A, inter=I, hidden_dropout=p_h, attn_dropout=p_a, seed=seed,
                       layer_index=layer_index, w_qkv=W["qkv"].data_ptr(), w_attn_out=W["o"].data_ptr(), w_inter=W["i"].data_ptr(),
                       w_out=W["out"].data_ptr(), b_qkv=bvec["qkv"].data_ptr(), b_attn_out=bvec["o"].data_ptr(),
                       ln1_gamma=ln["g1"].data_ptr(), ln1_beta=ln["b1"].data_ptr(), b_inter=bvec["i"].data_ptr(),
                       b_out=bvec["out"].data_ptr(), ln2_gamma=ln["g2"].data_ptr(), ln2_beta=ln["b2"].data_ptr(),
                       mask_bias=mbias.data_ptr())
    a = _lib.LayerActs(**{k: t.data_ptr() for k, t in acts.items()})
    _lib.check(L.vb_layer_fwd(ctypes.byref(d), ctypes.c_void_p(x.data_ptr()), ctypes.c_void_p(y.data_ptr()), ctypes.byref(a), st), "fwd")
    dy = rnd(Mr, H).to(bf)
    z = lambda *s: torch.zeros(*s, device=dev, dtype=f32)
    G = dict(dw_qkv=z(3 * H, H), db_qkv=z(3 * H), dw_attn_out=z(H, H), db_attn_out=z(H), dln1_gamma=z(H), dln1_beta=z(H),
             dw_inter=z(I, H), db_inter=z(I), dw_out=z(H, I), db_out=z(H), dln2_gamma=z(H), dln2_beta=z(H))
    sc = dict(d_pre=e(Mr, H), d_pre_drop=e(Mr, H), d_big=e(Mr, max(I, 3 * H)), d_x1=e(Mr, H), d_ctx=e(Mr, H), drow=e(B, A, S, dt=f32))
    dx = e(Mr, H)
    g_ = _lib.LayerGrads(**{k: t.data_ptr() for k, t in G.items()})
    s_ = _lib.LayerScratch(**{k: t.data_ptr() for k, t in sc.items()})
    _lib.check(L.vb_layer_bwd(ctypes.byref(d), ctypes.c_void_p(x.data_ptr()), ctypes.byref(a), ctypes.c_void_p(dy.data_ptr()),
                              ctypes.c_void_p(dx.data_ptr()), ctypes.byref(g_), ctypes.byref(s_), st), "bwd")
    torch.cuda.synchronize()

    # ---- the same masks ----
    nkb = (S + 63) // 64
    words = keep.view(torch.int64).view(2, B * A, nkb * 64, nkb)[0]
    bits = ((words.unsqueeze(-1) >> torch.arange(64, device=dev)) & 1).reshape(B * A, nkb * 64, nkb * 64)[:, :S, :S]
    keep_a = bits.view(B, A, S, S).float()
    n_a = int(p_a * 256.0 + 0.5)
    s_a = 256.0 / (256.0 - n_a)
    assert abs(keep_a.mean().item() - (1 - n_a / 256.0)) < 1e-2
    k1, s1 = hidden_keep(seed, layer_index * 8 + 1, Mr, H, p_h, dev)
    k2, s2 = hidden_keep(seed, layer_index * 8 + 2, Mr, H, p_h, dev)
    assert abs(k1.float().mean().item() - (1 - 26 / 256)) < 1e-2

    # ---- reference math (M.py:231-341), fp32, bf16-rounded weights, the library's masks ----
    P = {k: v.float().requires_grad_(True) for k, v in W.items()}
    Bv = {k: v.clone().requires_grad_(True) for k, v in bvec.items()}
    Ln = {k: v.clone().requires_grad_(True) for k, v in ln.items()}
    xr = x.float().requires_grad_(True)

    def lnorm(t, g, b):
        u = t.mean(-1, keepdim=True)
        v = (t - u).pow(2).mean(-1, keepdim=True)
        return g * ((t - u) / torch.sqrt(v + 1e-12)) + b

    qkv = xr @ P["qkv"].t() + Bv["qkv"]
    q, k, v = qkv.view(B, S, 3, A, 64).permute(2, 0, 3, 1, 4)
    probs = torch.softmax(q @ k.transpose(-1, -2) / 8.0 + mbias[:, None, None, :], -1) * keep_a * s_a      # M.py:241-251
    ctx = (probs @ v).permute(0, 2, 1, 3).reshape(Mr, H)
    x1 = lnorm((ctx @ P["o"].t() + Bv["o"]) * k1.float() * s1 + xr, Ln["g1"], Ln["b1"])                       # M.py:271-273
    u = x1 @ P["i"].t() + Bv["i"]
    h = u * 0.5 * (1.0 + torch.erf(u / math.sqrt(2.0)))                                                      # M.py:56-61
    yr = lnorm((h @ P["out"].t() + Bv["out"]) * k2.float() * s2 + x1, Ln["g2"], Ln["b2"])                     # M.py:316-318
    yr.backward(dy.float())

    def rel(a_, b_):
        return ((a_.float() - b_.float()).abs().max() / b_.float().abs().max().clamp_min(1e-9)).item()

    def relnorm(a_, b_):
        return ((a_.float() - b_.float()).norm() / b_.float().norm().clamp_min(1e-12)).item()

    assert rel(y, yr) < 2.5e-2, f"layer output: {rel(y, yr)}"
    assert relnorm(dx, xr.grad) < 2.5e-2, f"dx: {relnorm(dx, xr.grad)}"
    pairs = [("dw_qkv", P["qkv"]), ("db_qkv", Bv["qkv"]), ("dw_attn_out", P["o"]), ("db_attn_out", Bv["o"]),
             ("dln1_gamma", Ln["g1"]), ("dln1_beta", Ln["b1"]), ("dw_inter", P["i"]), ("db_inter", Bv["i"]),
             ("dw_out", P["out"]), ("db_out", Bv["out"]), ("dln2_gamma", Ln["g2"]), ("dln2_beta", Ln["b2"])]
    for name, ref in pairs:
        r = relnorm(G[name], ref.grad)
        assert r < 2.5e-2, f"{name}: relative gradient error {r}"


def test_side_stream_mask_generation_keeps_train_mode_parity():
    """The opt-in dropout-mask generation on a side stream under the QKV GEMM (VB_MASK_OVERLAP=1) must give the same train-mode
    parity (the GEMM variants are covered by test_kernels_gpu.py::test_gemm_kernel_variants): the switch is read once per
    process, so the parity test reruns in a subprocess."""
    import os, subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, VB_MASK_OVERLAP="1")
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-m", "gpu", "-q", "-k", "not side_stream"],
                       env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
