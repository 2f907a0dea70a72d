"""GPU: the attention kernels with a persistent item loop — attention_tcp.cu (forward), attention_bwd_tc.cu (v1) and
attention_bwd_tc2.cu (v2) — at production occupancy and at every tile-size boundary, with every dispatch path run on the same
inputs and checked against one float64 reference.

A persistent kernel launches min(n_items, #SMs) CTAs and each CTA walks a contiguous range of items, so a test with fewer
items than SMs never crosses an item boundary inside a CTA: stage / phase parity, per-item staging (bias strips and LUT rows in
the forward, lse / delta in the backward) and the late read-out of finished accumulators into the next item are only exercised
with more items than SMs.  Shapes here are derived from the device's SM count.

Errors are measured per (batch, head) item — max |kernel - reference| over the item divided by the item's max |reference| —
so that one wrong item cannot hide under the global maximum of a large tensor.  Every case prints the worst and median item
error and where the worst one sits (run with -s).  A sample with a single valid key has dQ = dK = 0 exactly (dS = P (dP - delta)
vanishes for P = 1), so an item's scale is floored at ITEM_FLOOR x the largest item's (and, where the whole tensor vanishes at
S = 1, at a small absolute scale).

Bars (FWD_BARS, BWD_BARS): P and dS are rounded to bf16 on the tensor cores (2^-9 relative each), the bias is kept as fp16
(x log2 e) except in the per-tile forward, and outputs and gradients are rounded to bf16.
Different paths agree only within that rounding (DESIGN.md 4.6), so paths are compared with the reference, never bitwise
with each other; the one bitwise comparison is of a kernel with itself (determinism, cluster launch).

Run as a script (`python tests/test_gpu_attention_occupancy.py --cluster-child OUT`) it computes the cluster-launch outputs in a
fresh process: OPB_ATTN_CLUSTER_LAUNCH is read once per process (common.cuh, launch_maybe_cluster)."""
import math
import os
import subprocess
import sys
from types import SimpleNamespace

import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
Q_SCALE = 0.125
ITEM_FLOOR = 0.05
NAN = float("nan")

# worst-item bars per path (relative to the item's scale; lse absolute, natural log): ~1.5x the worst item measured over this
# file's cases on a B200 (148 SMs, 1000 W power limit).  The persistent forward keeps the bias as fp16 (lse within 1.3e-3); the
# per-tile one's lse is within 4e-6, its out / LayerNorm sums of squares within 7.8e-3.  Backward: dQ / dK / dV within 8.1e-3
# on every path, dbias within 1.4e-3.
FWD_BARS = {"tcp": {"out": 6e-3, "lse": 2e-3, "ln_sum": 1e-3, "ln_sumsq": 3e-3},
            "tc": {"out": 1.1e-2, "lse": 1e-5, "ln_sum": 2.5e-3, "ln_sumsq": 1.2e-2}}
BWD_BARS = {"dq": 1.1e-2, "dk": 1e-2, "dv": 1.2e-2, "dbias": 2.5e-3}

# tcp forward: nb16 = ceil(S / 16) -> instantiation <2, 4, 6, 9, 13, 14>; both sides of every edge, the 'vl' length 214, and 225
# (first length on the per-tile kernel)
FWD_S = [1, 16, 17, 32, 33, 64, 65, 96, 97, 144, 145, 208, 209, 214, 224, 225]
# v2 backward: key tiles of 128 x query quarters of 64 -> (n_kt, n_q) = (1, 1), (1, 2), (2, 3), (2, 4); v1 backward: query half
# qh = 48 / 80 / 112 / 2 x 112 at S <= 48 / 80 / 112 / 224; 225 is past both (dense entry point: the mma.sync pair)
BWD_S = [1, 8, 16, 17, 48, 49, 63, 64, 65, 80, 81, 112, 113, 127, 128, 129, 192, 193, 214, 224, 225]
# key-padding lengths, cycled over the batch: one key; one full key tile (the second one fully masked); one key into the second
# tile; the full length ('ragged') or just short of it ('short': then the last keys are padded in every sample)
PADS = [None, "ragged", "short"]

FWD_PATHS = (("tcp", {}), ("tc", {"OPB_ATTN_PERSIST": "0"}))
# (name, bias form, switches): v2 and v1 behind opb_attention_bwd_t (transposed tables), v1 and the mma.sync pair behind
# opb_attention_bwd (dense tables)
BWD_PATHS = (("v2", "t", {}), ("v1_t", "t", {"OPB_ATTN_BWD_V": "1"}), ("v1", "dense", {}),
             ("mma", "dense", {"OPB_ATTN_BWD_TC": "0"}))


@pytest.fixture(scope="module")
def K():
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    from one_peace_b200 import kernels
    return kernels


def sm_count():
    return torch.cuda.get_device_properties(0).multi_processor_count


# ----------------------------------------------------------------------------------------------------------------- inputs
def key_pad_lengths(pattern, B, S):
    if pattern is None:
        return [S] * B
    if pattern == "ragged":
        cyc, top = (129, 1, 128, S), S
    else:
        cyc, top = (129, 1, 128, S - 5), max(1, S - 1)
    return [max(1, min(top, cyc[b % 4])) for b in range(B)]


def make_case(K, B, S, H, kind, pad, seed):
    """bf16 qkv / d_out, the relative-position bias in the LUT form the tcgen05 forward takes and as the dense (H,S,S) table
    it stands for (built from the same LUT, as in test_gpu_kernels.py::test_attention_tc), and the key padding."""
    import restated as R
    from one_peace_b200 import relpos
    D = H * 64
    g = torch.Generator(device="cuda").manual_seed(seed)
    qkv = (torch.randn(B * S, 3 * D, device="cuda", generator=g) * 0.5).bfloat16()
    d_out = torch.randn(B * S, D, device="cuda", generator=g).bfloat16()
    if kind == "text":
        bucket = R.make_token_bucket_position(256)[:S, :S]
        codes, ntab = relpos.text_codes(S), 514
    else:
        w = int(round((S - 1) ** 0.5))
        assert w * w + 1 == S
        bucket, codes, ntab = R.make_image_bucket_position(w), relpos.image_codes(S, w), (2 * w - 1) ** 2 + 3
    table = torch.randn(ntab, H, device="cuda", generator=g)
    lut_idx, crow, ccol = (torch.from_numpy(a).cuda() for a in relpos.build_lut_index(bucket.numpy(), codes))
    rp = K.RelPosBias(lut=K.relpos_lut_build(table, lut_idx), code_row=crow, code_col=ccol)
    dense = rp.lut[:, (crow[:S, None] - ccol[None, :S]).long()].contiguous()
    assert torch.equal(dense, table[bucket.cuda()].permute(2, 0, 1))
    s_pad = (S + 7) // 8 * 8
    dense_pad = torch.zeros(H, S, s_pad, device="cuda")
    dense_pad[..., :S] = dense
    lens = key_pad_lengths(pad, B, S)
    kp = None
    if pad is not None:
        kp = torch.zeros(B, S, dtype=torch.uint8, device="cuda")
        for b, n in enumerate(lens):
            kp[b, n:] = 1
    return SimpleNamespace(B=B, S=S, H=H, D=D, qkv=qkv, d_out=d_out, rp=rp, dense=dense, dense_pad=dense_pad, kp=kp, lens=lens)


# -------------------------------------------------------------------------------------------------------------- reference
def attention_ref64(qkv, bias_dense, key_pad, B, S, H, d_out=None, q_scale=Q_SCALE):
    """float64 attention on the bf16 operands (q in `qkv` is stored scaled, multihead_attention.py:107-115), differentiated by
    torch autograd.  Returns per-item tensors: out [B,H,S,64], lse [B,H,S] and, given d_out, dq (times q_scale, as the kernels
    write it), dk, dv [B,H,S,64] and dbias [H,S,S] (summed over the batch).

    The gradients are those of the backward's contract: the kernels are handed the bf16 output and take
    delta = rowsum(dO * O) from it (attn_delta, as flash attention does).  Softmax's adjoint is P * (dP - delta); holding the
    normaliser fixed, autograd of sum(dO * P V) - sum(delta * P) with that delta as a constant gives exactly this, and the
    true gradient when O is exact.  (With exact O instead, samples of a few keys differ by up to 3e-2 per item — the same
    for every kernel: dP - delta is then a small difference.)"""
    grad = d_out is not None
    x = qkv.double().requires_grad_(grad)
    bias = bias_dense.double().requires_grad_(grad)
    q, k, v = x.view(B, S, 3, H, 64).permute(2, 0, 3, 1, 4)
    s = q @ k.transpose(-1, -2) + bias
    if key_pad is not None:
        s = s.masked_fill(key_pad.bool()[:, None, None, :], float("-inf"))
    lse = torch.logsumexp(s, -1)
    o = torch.softmax(s, -1) @ v
    r = {"out": o.detach(), "lse": lse.detach()}
    if grad:
        do = d_out.double().view(B, S, H, 64).transpose(1, 2)
        p = torch.exp(s - lse.detach()[..., None])
        delta = (do * o.detach().bfloat16().double()).sum(-1, keepdim=True)
        (((p @ v) * do).sum() - (p * delta).sum()).backward()
        dq, dk, dv = x.grad.view(B, S, 3, H, 64).permute(2, 0, 3, 1, 4)
        r.update(dq=dq * q_scale, dk=dk, dv=dv, dbias=bias.grad)
    return r


def items(t, B, S, H):
    """[B*S, H*64] row-major activations -> [B, H, S, 64]"""
    return t.view(B, S, H, 64).transpose(1, 2)


def item_errors(got, want, lead=2, relative=True, scale=None, floor=0.0):
    """per-item error over the `lead` leading dims: max |got - want| / max(item's max |want|, ITEM_FLOOR x largest item's,
    `floor`), or the absolute error.  Returns (worst, median, index of the worst item); a NaN (an element no kernel wrote) is
    the worst."""
    shape = tuple(want.shape[:lead])
    g = got.double().reshape(math.prod(shape), -1)
    w = want.double().reshape(math.prod(shape), -1)
    err = (g - w).abs().amax(1)
    if relative:
        sc = (w.abs() if scale is None else scale.double().reshape(math.prod(shape), -1)).amax(1)
        err = err / sc.clamp_min(max(ITEM_FLOOR * sc.max().item(), floor, 1e-30))
    err = torch.nan_to_num(err, nan=float("inf"))
    i = int(err.argmax())
    idx = tuple(int(v) for v in torch.unravel_index(torch.tensor(i), shape))
    return err[i].item(), err.median().item(), idx


class Report:
    """collects every comparison of a case, prints it, fails at the end with all violations"""

    def __init__(self, label):
        self.label, self.bad = label, []

    def occupancy(self, kernel, n_items):
        sms = sm_count()
        grid = min(n_items, sms)
        print(f"\n{self.label} {kernel}: n_items {n_items} sms {sms} items per CTA {n_items // grid}-{-(-n_items // grid)}", end="")

    def check(self, path, name, got, want, bar, **kw):
        worst, med, idx = item_errors(got, want, **kw)
        print(f"\n  {self.label} {path} {name}: worst {worst:.3e} median {med:.3e} at {idx} (bar {bar:.2g})", end="")
        if not worst < bar:
            self.bad.append(f"{path} {name}: worst item {idx} {worst:.3e} >= {bar:.2g}")

    def require(self, path, what, ok):
        if not ok:
            self.bad.append(f"{path}: {what}")

    def done(self):
        print()
        assert not self.bad, f"{self.label}: " + "; ".join(self.bad)


# ---------------------------------------------------------------------------------------------------------------- kernels
def run_forward(K, c):
    """tcgen05 forward into NaN-filled out / lse / LayerNorm partials (whatever the kernel does not write stays NaN)"""
    B, S, H = c.B, c.S, c.H
    out = torch.full((B * S, c.D), NAN, device="cuda", dtype=torch.bfloat16)
    lse = torch.full((B * H * S,), NAN, device="cuda")
    part = torch.full((H * B * S * 2,), NAN, device="cuda")
    K.attention_tc(c.qkv, c.rp, c.kp, B, S, H, out=out, ln_stats=part, lse=lse)
    torch.cuda.synchronize()
    return out, lse, part


def run_backward(K, c, form, out, lse):
    """one backward into a NaN-filled dqkv; returns (dqkv, dbias (H,S,S), the raw gradient table)"""
    B, S, H = c.B, c.S, c.H
    dqkv = torch.full((B * S, 3 * c.D), NAN, device="cuda", dtype=torch.bfloat16)
    dbias = torch.zeros_like(c.dense_pad)
    if form == "t":
        raw = torch.zeros(H, K.BIAS_T_KEYS, K.BIAS_T_Q, device="cuda")
        K.attention_bwd_t(c.qkv, out, c.d_out, K.relpos_bias_transpose(c.dense_pad), c.kp, lse, dqkv, raw, B, S, H, Q_SCALE)
        K.relpos_dbias_fold(raw, dbias)
    else:
        K.attention_bwd(c.qkv, out, c.d_out, c.dense_pad, c.kp, lse, dqkv, dbias, B, S, H, Q_SCALE)
        raw = dbias
    torch.cuda.synchronize()
    return dqkv, dbias[..., :S], raw


def check_forward(K, monkeypatch, rep, c, ref):
    B, S, H = c.B, c.S, c.H
    if S <= 224:
        rep.occupancy("tcp", B * H * (-(-S // 128)))
    for path, env in FWD_PATHS:
        if path == "tcp" and S > 224:
            continue
        with monkeypatch.context() as m:
            for k, v in env.items():
                m.setenv(k, v)
            out, lse, part = run_forward(K, c)
        bar = FWD_BARS[path]
        rep.check(path, "out", items(out, B, S, H), ref["out"], bar["out"])
        rep.check(path, "lse", lse.view(B, H, S), ref["lse"], bar["lse"], relative=False)
        # per-head LayerNorm partials (sum, sum of squares) of the fp32 output rows before rounding; |sum| <= sqrt(64 sumsq)
        p = part.view(H, B, S, 2).transpose(0, 1)
        ref_sq = (ref["out"] ** 2).sum(-1)
        rep.check(path, "ln_sum", p[..., 0], ref["out"].sum(-1), bar["ln_sum"], scale=(64 * ref_sq).sqrt())
        rep.check(path, "ln_sumsq", p[..., 1], ref_sq, bar["ln_sumsq"])


def check_backward(K, monkeypatch, rep, c, ref):
    """every backward path on the kernels' inputs of the forward: reference output (bf16) and log-sum-exp (fp32)"""
    B, S, H, D = c.B, c.S, c.H, c.D
    out = ref["out"].transpose(1, 2).reshape(B * S, D).bfloat16()
    lse = ref["lse"].float().reshape(-1).contiguous()
    rep.occupancy("v1/v2", B * H)
    pad_rows = c.kp.bool() if c.kp is not None else torch.zeros(B, S, dtype=torch.bool, device="cuda")
    all_pad = pad_rows.all(0)                                          # keys padded in every sample
    # dQ, dK and dbias vanish identically at S = 1 (P = 1): there the scale is an absolute one, from dV (which never vanishes)
    tiny = 1e-3 * ref["dv"].abs().max().item()
    for path, form, env in BWD_PATHS:
        with monkeypatch.context() as m:
            for k, v in env.items():
                m.setenv(k, v)
            if form == "t" and S > 224:                                # S <= 224 only: refused, not computed
                with pytest.raises(RuntimeError):
                    K.attention_bwd_t(c.qkv, out, c.d_out, None, c.kp, lse, torch.empty_like(c.qkv), None, B, S, H, Q_SCALE)
                continue
            dqkv, dbias, raw = run_backward(K, c, form, out, lse)
        g = dqkv.view(B, S, 3, H, 64)
        for i, name in enumerate(("dq", "dk", "dv")):
            rep.check(path, name, g[:, :, i].transpose(1, 2), ref[name], BWD_BARS[name], floor=tiny)
        rep.check(path, "dbias", dbias, ref["dbias"], BWD_BARS["dbias"], lead=1, floor=tiny)
        rep.require(path, "dK / dV rows of padded keys are not exactly zero", torch.count_nonzero(g[:, :, 1:][pad_rows]) == 0)
        if form == "t":
            rep.require(path, "dbias_t: keys padded in every sample got a gradient", torch.count_nonzero(raw[:, :S][:, all_pad]) == 0)
            rep.require(path, "dbias_t: written outside the S x S corner",
                        torch.count_nonzero(raw[:, S:]) == 0 and torch.count_nonzero(raw[:, :, S:]) == 0)
        else:
            rep.require(path, "dbias: keys padded in every sample got a gradient", torch.count_nonzero(raw[:, :, :S][..., all_pad]) == 0)
            rep.require(path, "dbias: written past column S", torch.count_nonzero(raw[..., S:]) == 0)


def edge_shape(shape, S):
    """'small': 4 samples x 2 heads (one item per CTA); 'multi': 2-3 items per CTA (5-6 forward tiles past S = 128)"""
    if shape == "small":
        return 4, 2
    H = 8
    return 4 * -(-5 * sm_count() // (2 * 4 * H)), H


# ------------------------------------------------------------------------------------------------------------------ tests
@pytest.mark.parametrize("pad", PADS)
@pytest.mark.parametrize("shape", ["small", "multi"])
@pytest.mark.parametrize("S", FWD_S)
def test_forward_seq_edges(K, monkeypatch, S, shape, pad):
    B, H = edge_shape(shape, S)
    c = make_case(K, B, S, H, "text", pad, seed=S * 10 + len(shape))
    ref = attention_ref64(c.qkv, c.dense, c.kp, B, S, H)
    rep = Report(f"fwd S={S} B={B} H={H} pad={pad}")
    check_forward(K, monkeypatch, rep, c, ref)
    rep.done()


@pytest.mark.parametrize("pad", PADS)
@pytest.mark.parametrize("shape", ["small", "multi"])
@pytest.mark.parametrize("S", BWD_S)
def test_backward_seq_edges(K, monkeypatch, S, shape, pad):
    B, H = edge_shape(shape, S)
    c = make_case(K, B, S, H, "text", pad, seed=S * 10 + len(shape) + 1)
    ref = attention_ref64(c.qkv, c.dense, c.kp, B, S, H, d_out=c.d_out)
    rep = Report(f"bwd S={S} B={B} H={H} pad={pad}")
    check_backward(K, monkeypatch, rep, c, ref)
    rep.done()


# (B, S, H, kind) from the SM count: sms + 1 and 2 sms - 1 items (CTAs with one and two items side by side), the production
# vision shape (~10 backward items and ~21 forward tiles per CTA), and H = 128 (the kernels' limit) with small B, whose CTA
# ranges cross a (head, q-tile) boundary almost everywhere
OCCUPANCY = {
    "sms+1": lambda sms: (sms + 1, 100, 1, "text"),
    "2sms-1": lambda sms: (2 * sms - 1, 150, 1, "text"),
    "production": lambda sms: (64, 197, 24, "image"),
    "wide_b3": lambda sms: (3, 197, 128, "image"),
    "wide_b1": lambda sms: (1, 224, 128, "text"),
}


@pytest.mark.parametrize("pad", [None, "ragged"])
@pytest.mark.parametrize("case", list(OCCUPANCY))
def test_occupancy(K, monkeypatch, case, pad):
    B, S, H, kind = OCCUPANCY[case](sm_count())
    c = make_case(K, B, S, H, kind, pad, seed=len(case) * 100 + S)
    ref = attention_ref64(c.qkv, c.dense, c.kp, B, S, H, d_out=c.d_out)
    rep = Report(f"{case} B={B} S={S} H={H} pad={pad}")
    check_forward(K, monkeypatch, rep, c, ref)
    check_backward(K, monkeypatch, rep, c, ref)
    rep.done()


def test_repeat_calls_bitwise_equal(K, monkeypatch):
    """every output element is written by exactly one CTA (dbias_t, a red.global.add sum, is left out)"""
    B, S, H = 64, 197, 24
    c = make_case(K, B, S, H, "image", "ragged", seed=5)
    a, b = run_forward(K, c), run_forward(K, c)
    assert all(torch.equal(x, y) for x, y in zip(a, b))
    out, lse = a[0], a[1]
    for path, form, env in BWD_PATHS[:2]:
        with monkeypatch.context() as m:
            for k, v in env.items():
                m.setenv(k, v)
            d1, d2 = run_backward(K, c, form, out, lse)[0], run_backward(K, c, form, out, lse)[0]
        assert torch.equal(d1, d2), path


def cluster_case_outputs(K, setenv):
    """forward (tcp) and both transposed-table backwards (v2, then v1) of one seeded multi-item shape, as CPU tensors"""
    c = make_case(K, 16, 197, 24, "image", "ragged", seed=11)
    out, lse, part = run_forward(K, c)
    r = {"out": out, "lse": lse, "ln": part, "dqkv_v2": run_backward(K, c, "t", out, lse)[0]}
    setenv("OPB_ATTN_BWD_V", "1")
    r["dqkv_v1"] = run_backward(K, c, "t", out, lse)[0]
    return {k: v.cpu() for k, v in r.items()}


def test_cluster_launch_matches_plain_launch(K, monkeypatch, tmp_path):
    """OPB_ATTN_CLUSTER_LAUNCH=1 (one-CTA clusters through cudaLaunchKernelEx) computes bit for bit what the plain launch does.
    The switch is cached at first use, so the cluster arm runs in a child process of its own."""
    if os.environ.get("OPB_ATTN_CLUSTER_LAUNCH", "0") == "1":
        pytest.skip("this process already launches the attention kernels as clusters")
    dump = tmp_path / "cluster.pt"
    env = dict(os.environ, OPB_ATTN_CLUSTER_LAUNCH="1")
    for k in ("OPB_ATTN_BWD_V", "OPB_ATTN_BWD_TC", "OPB_ATTN_PERSIST"):
        env.pop(k, None)
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [os.path.abspath(__file__), "--cluster-child", str(dump)]
    proc = subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True, timeout=900)
    assert proc.returncode == 0, proc.stdout[-2000:] + proc.stderr[-4000:]
    got = torch.load(dump)
    want = cluster_case_outputs(K, monkeypatch.setenv)
    for k in want:
        assert torch.equal(got[k], want[k]), k


if __name__ == "__main__":
    if len(sys.argv) == 3 and sys.argv[1] == "--cluster-child":
        for p in (ROOT, os.path.join(ROOT, "oracle")):
            sys.path.insert(0, p)
        from one_peace_b200 import kernels
        torch.save(cluster_case_outputs(kernels, os.environ.__setitem__), sys.argv[2])
    else:
        sys.exit(f"usage: {sys.argv[0]} --cluster-child OUT.pt")
