"""The three decoder attention kernels against a float64 reference of the same operation, and the engine's decoder step over the
whole 448-position cache on every step path.

  * self_attn_kernel (csrc/decode_stream.cu) through bw_op_self_attn: positions on both sides of the 128-key chunk boundaries of its
    online softmax, every output type, both 16-bit builds, ancestry tables, the batched path's in-kernel cache append.
  * cross_attn_kernel<1 | 8> (split) and cross_attn_stream_kernel<1..5 | 8> through bw_op_cross_attn: every beam count, key lengths
    with empty split blocks and ragged streaming tiles, the word-timestamp score capture.
  * the engine's decoder step (persistent kernel, per-op kernels, batched step with either cross-attention kernel) teacher-forced
    over all 448 positions against the HF model in fp32, greedy to the end of the cache, and the alignment scores it records.

References are computed in float64 from the 16-bit-rounded K / V and the fp32 q the kernel sees.  Every bound is printed beside
the value measured on the B200 (`-s`); the bounds are about 3x the measured maxima (profiles/r3_decoder_attn.log).
"""
import ctypes as C
import json
import os

import numpy as np
import pytest
import torch

from tests.conftest import GOLD

pytestmark = pytest.mark.gpu

E16 = {"bf16": (torch.bfloat16, 0), "fp16": (torch.float16, 1)}
HALF_ULP = {"bf16": 2.0 ** -8, "fp16": 2.0 ** -11}  # relative half-ulp of one rounding to the 16-bit type
BW_CHECK_RC = -2  # what a failed host-side argument check returns (common.cuh BW_CHECK)

# bounds, as multiples of max|V| (outputs) or of |q| |k| (alignment scores); 16-bit outputs: error beyond one rounding of the reference.
# Measured on a B200 (1000 W): self-attention 1.4e-7, cross-attention 4.3e-7 (streaming) / 1.6e-7 (split), alignment scores 2.4e-7,
# needles exact (0); profiles/r3_decoder_attn.log
SELF_BOUND = 5e-7
CROSS_BOUND = 1.5e-6
NEEDLE_BOUND = 1e-7
ALIGN_BOUND = 1e-6

_MEASURED = {}


def _note(key, value, bound):
    v, _ = _MEASURED.get(key, (0.0, bound))
    _MEASURED[key] = (max(v, float(value)), bound)


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    if _MEASURED:
        print("\n[decoder attention] measured maximum vs bound")
        for key in sorted(_MEASURED):
            v, b = _MEASURED[key]
            print(f"  {key:<48s} {v:.3e}  (bound {b:.1e})")


def _lib():
    from thewhisper_b200 import _lib

    return _lib, _lib.load()


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _pos_dev(pos, dev):
    return torch.tensor([pos], dtype=torch.int32, device=dev)


def _out_err(got, ref, vmax, dtype):
    """max error in units of max|V|; a 16-bit output is allowed one rounding of the reference on top"""
    d = (got.double() - ref).abs()
    if got.dtype != torch.float32:
        d = (d - HALF_ULP[dtype] * ref.abs()).clamp_min(0.0)
    return d.max().item() / vmax


# ------------------------------------------------------------------------------------------------------------------
# a. self-attention op
# ------------------------------------------------------------------------------------------------------------------
TMAX = 448
SELF_POS = [0, 1, 7, 126, 127, 128, 129, 143, 144, 255, 256, 300, 447]


def _self_attn(qkv, kc, vc, pos, Q, H, dtype, out_f32, anc=None, nsplit=0, bias=None, alpha=1.0, append=False):
    L, lib = _lib()
    D = H * 64
    out = torch.full((Q, D), float("nan"), dtype=torch.float32 if out_f32 else E16[dtype][0], device=qkv.device)
    rc = lib.bw_op_self_attn(_ptr(qkv), nsplit, _ptr(bias), alpha, _ptr(kc), _ptr(vc), _ptr(anc), int(append), _ptr(out), int(out_f32),
                             _ptr(_pos_dev(pos, qkv.device)), Q, H, TMAX, E16[dtype][1], _stream())
    L.check(rc)
    torch.cuda.synchronize()
    return out


def _ref_self(q, kc, vc, pos, Q, H, anc=None):
    """q [Q, D] float64; kc / vc [Q, Tmax, D] 16-bit -> [Q, D] float64 (keys 0..pos of the slot anc[q, s])"""
    n = pos + 1
    slots = anc[:, :n].long() if anc is not None else torch.arange(Q, device=q.device)[:, None].expand(Q, n)
    s_idx = torch.arange(n, device=q.device)[None, :].expand(Q, n)
    K = kc[slots, s_idx].double().view(Q, n, H, 64)
    V = vc[slots, s_idx].double().view(Q, n, H, 64)
    sc = torch.einsum("qhd,qshd->qhs", q.view(Q, H, 64), K)
    p = torch.softmax(sc, dim=-1)
    return torch.einsum("qhs,qshd->qhd", p, V).reshape(Q, H * 64)


def _self_case(Q, H, pos, mode, g, dev, dtype):
    """q [Q, D] fp32 and a cache [Q, Tmax, D] whose rows beyond pos are NaN (a key past the causal end would poison the output).
    mode: random / rising / falling scores along the key axis, or ("needle", j): key j scores 40 above every other key."""
    D = H * 64
    n = pos + 1
    et = E16[dtype][0]
    q = torch.randn(Q, D, generator=g) * 0.3
    K = torch.randn(Q, TMAX, D, generator=g) * 0.5
    V = torch.randn(Q, TMAX, D, generator=g)
    if mode in ("rising", "falling"):
        # key s gets a score of about target[s] (+- 0.5): q is one direction per head, K carries the ramp along it
        q = torch.zeros(Q, D)
        q.view(Q, H, 64)[:, :, 0] = 2.0
        ramp = torch.linspace(-3.0, 3.0, n) if mode == "rising" else torch.linspace(3.0, -3.0, n)
        K.view(Q, TMAX, H, 64)[:, :n, :, 0] = ramp[None, :, None]
        K.view(Q, TMAX, H, 64)[:, :n, :, 1:] *= 0.1
    elif isinstance(mode, tuple):
        j = mode[1]
        q = torch.zeros(Q, D)
        q.view(Q, H, 64)[:, :, 0] = 11.0
        K.view(Q, TMAX, H, 64)[:, :n, :, 0] = torch.rand(Q, n, H, generator=g) * 0.1
        K.view(Q, TMAX, H, 64)[:, j, :, 0] = 4.0
    K[:, n:] = float("nan")
    V[:, n:] = float("nan")
    return q.to(dev), K.to(et).to(dev), V.to(et).to(dev)


@pytest.mark.parametrize("dtype", ["bf16", "fp16"])
@pytest.mark.parametrize("Q,H", [(1, 1), (3, 2), (10, 20), (64, 6)])
@pytest.mark.parametrize("pos", SELF_POS)
def test_self_attn_op(cuda, pos, Q, H, dtype):
    """Outputs fp32 and 16-bit; random / rising / falling scores (the running max grows in every chunk / sits in chunk 0); ancestry
    tables (anc[q, pos] == q); needles at keys 0, 127, 128, 129, pos-1 and pos must return that key's V row."""
    g = torch.Generator(device="cpu").manual_seed(pos * 1000 + Q * 10 + H)
    D = H * 64
    for mode in ("random", "rising", "falling"):
        q, kc, vc = _self_case(Q, H, pos, mode, g, cuda, dtype)
        vmax = vc[:, : pos + 1].float().abs().max().item()
        ancs = [None]
        if mode == "random":
            anc = torch.randint(0, Q, (Q, TMAX), generator=g, dtype=torch.int32)
            anc[:, pos] = torch.arange(Q, dtype=torch.int32)
            ancs.append(anc.to(cuda))
        for anc in ancs:
            ref = _ref_self(q.double(), kc, vc, pos, Q, H, anc)
            qkv = torch.zeros(Q, 3 * D, device=cuda)
            qkv[:, :D] = q
            for out_f32 in (True, False):
                out = _self_attn(qkv, kc, vc, pos, Q, H, dtype, out_f32, anc=anc)
                err = _out_err(out, ref, vmax, dtype)
                _note(f"self_attn {dtype} {'fp32' if out_f32 else '16-bit'} out", err, SELF_BOUND)
                assert err <= SELF_BOUND, (mode, anc is not None, out_f32, err)
    for j in sorted({0, 127, 128, 129, pos - 1, pos}):
        if not 0 <= j <= pos:
            continue
        q, kc, vc = _self_case(Q, H, pos, ("needle", j), g, cuda, dtype)
        qkv = torch.zeros(Q, 3 * D, device=cuda)
        qkv[:, :D] = q
        want = vc[:, j].double()
        vmax = vc[:, : pos + 1].float().abs().max().item()
        for out_f32 in (True, False):
            out = _self_attn(qkv, kc, vc, pos, Q, H, dtype, out_f32)
            err = _out_err(out, want, vmax, dtype)
            _note(f"self_attn {dtype} needle", err, NEEDLE_BOUND)
            assert err <= NEEDLE_BOUND, (j, out_f32, err)


@pytest.mark.parametrize("dtype", ["bf16", "fp16"])
@pytest.mark.parametrize("nsplit", [1, 4])
@pytest.mark.parametrize("Q,H", [(1, 1), (3, 2), (10, 20), (64, 6)])
@pytest.mark.parametrize("pos", [0, 127, 128, 129, 300, 447])
def test_self_attn_append(cuda, pos, Q, H, nsplit, dtype):
    """Batched path: qkv holds nsplit raw partial sums; the kernel adds them in order (+ bias, q * alpha), writes k / v rounded to
    16 bit at row pos of the cache and attends over it.  Every other cache row is left as it was (sentinel fill)."""
    g = torch.Generator(device="cpu").manual_seed(7 + pos * 100 + Q * 10 + H + nsplit)
    D = H * 64
    et = E16[dtype][0]
    parts = (torch.randn(nsplit, Q, 3 * D, generator=g) * 0.4).to(cuda)
    bias = (torch.randn(3 * D, generator=g) * 0.2).to(cuda)
    alpha = 0.125
    kc = (torch.randn(Q, TMAX, D, generator=g) * 0.5).to(et).to(cuda)
    vc = torch.randn(Q, TMAX, D, generator=g).to(et).to(cuda)
    sentinel = torch.tensor(-777.0, dtype=et)
    kc[:, pos:] = sentinel.to(cuda)
    vc[:, pos:] = sentinel.to(cuda)
    kc0, vc0 = kc.clone(), vc.clone()
    for out_f32 in (True, False):
        kc.copy_(kc0)
        vc.copy_(vc0)
        out = _self_attn(parts, kc, vc, pos, Q, H, dtype, out_f32, nsplit=nsplit, bias=bias, alpha=alpha, append=True)
        # fp32 sum in split order, then + bias: the kernel's order, so the rounded row is exact
        acc = parts[0].clone()
        for s in range(1, nsplit):
            acc = acc + parts[s]
        acc = acc + bias
        assert torch.equal(kc[:, pos], acc[:, D:2 * D].to(et)), "k row"
        assert torch.equal(vc[:, pos], acc[:, 2 * D:].to(et)), "v row"
        mask = torch.ones(TMAX, dtype=torch.bool)
        mask[pos] = False
        assert torch.equal(kc[:, mask].view(torch.int16), kc0[:, mask].view(torch.int16)), "cache rows other than pos were written"
        assert torch.equal(vc[:, mask].view(torch.int16), vc0[:, mask].view(torch.int16))
        q = parts.double().sum(0)[:, :D] + bias.double()[:D]
        ref = _ref_self(q * alpha, kc, vc, pos, Q, H)
        vmax = vc[:, : pos + 1].float().abs().max().item()
        err = _out_err(out, ref, vmax, dtype)
        _note(f"self_attn {dtype} append", err, SELF_BOUND)
        assert err <= SELF_BOUND, (out_f32, err)


# ------------------------------------------------------------------------------------------------------------------
# b. cross-attention op
# ------------------------------------------------------------------------------------------------------------------
XSPLIT, MAXS = 12, 1536
CROSS_S = [1, 5, 11, 127, 128, 129, 250, 500, 750, 1499, 1500, 1536]
CH = 3  # heads; alignment capture: head 0 -> slot 1, head 1 -> none, head 2 -> slot 0
HEAD_SLOTS = [1, -1, 0]
HA, TCAP, STEP_BASE = 2, 4, 5


class _XScratch:
    def __init__(self, A, G, H, dev):
        self.part_o = torch.full((A * H * XSPLIT * G * 64,), float("nan"), device=dev)
        self.part_ml = torch.full((A * H * XSPLIT * G * 2,), float("nan"), device=dev)
        self.counters = torch.zeros(A * H, dtype=torch.int32, device=dev)


def _cross_attn(qin, nsplit, bias, alpha, kc, vc, A, G, H, S, dtype, out_f32, impl, scratch, align=None, head_slots=None, pos=None):
    L, lib = _lib()
    out = torch.full((A * G, H * 64), float("nan"), dtype=torch.float32 if out_f32 else E16[dtype][0], device=kc.device)
    pos_t = _pos_dev(pos, kc.device) if pos is not None else None
    rc = lib.bw_op_cross_attn(_ptr(qin), nsplit, _ptr(bias), alpha, _ptr(kc), _ptr(vc), _ptr(out), int(out_f32), _ptr(scratch.part_o),
                              _ptr(scratch.part_ml), _ptr(scratch.counters), A, G, H, S, _ptr(align), _ptr(head_slots), HA, TCAP,
                              STEP_BASE, _ptr(pos_t), impl, E16[dtype][1], _stream())
    return rc, out


def _ref_cross(q, kc, vc, A, G, H, S):
    """q [A*G, D] float64, kc / vc [A, H, S, 64] -> out [A*G, D] float64, raw scores [A, G, H, S] float64"""
    K, V = kc.double(), vc.double()
    qq = q.view(A, G, H, 64)
    sc = torch.einsum("aghd,ahsd->aghs", qq, K)
    out = torch.einsum("aghs,ahsd->aghd", torch.softmax(sc, dim=-1), V)
    return out.reshape(A * G, H * 64), sc


def _cross_case(A, G, S, mode, g, dev, dtype):
    D = CH * 64
    et = E16[dtype][0]
    kc = torch.randn(A, CH, S, 64, generator=g) * 0.5
    vc = torch.randn(A, CH, S, 64, generator=g)
    q = torch.randn(A * G, D, generator=g) * 0.3
    needles = None
    if mode == "rising":
        kc[..., 0] = torch.linspace(-3.0, 3.0, S)
        kc[..., 1:] *= 0.1
        q = torch.zeros(A * G, D)
        q.view(A * G, CH, 64)[:, :, 0] = 2.0 + 0.1 * torch.arange(G).repeat(A)[:, None]
    elif mode == "needle":
        # the needle of (audio a, beam g): key needles[a][g] is 4 along dim g, every other key ~0.05 there; q = 12 e_g: a gap of ~45
        cand = sorted({j for j in (0, 127, 128, 129, S - 2, S - 1) if 0 <= j < S})
        needles = [[cand[(a + g_) % len(cand)] for g_ in range(G)] for a in range(A)]
        kc[..., :8] = torch.randn(A, CH, S, 8, generator=g) * 0.05
        q = torch.zeros(A * G, D)
        for a in range(A):
            for g_, j in enumerate(needles[a]):
                kc[a, :, j, g_] = 4.0
                q.view(A, G, CH, 64)[a, g_, :, g_] = 12.0
    return q.to(dev), kc.to(et).to(dev), vc.to(et).to(dev), needles


def _q_input(q, nsplit, g, dev):
    """fp32 q as the engine's cross-q projection leaves it: final (nsplit 0) or nsplit raw partial sums with a bias and q_alpha"""
    if nsplit == 0:
        return q, None, 1.0, q.double()
    alpha = 0.125
    bias = torch.randn(q.shape[1], generator=g).to(dev) * 0.5
    parts = torch.randn(nsplit, *q.shape, generator=g).to(dev)
    parts[-1] = q / alpha - bias - parts[:-1].sum(0)
    eff = (parts.double().sum(0) + bias.double()) * alpha
    return parts.contiguous(), bias, alpha, eff


@pytest.mark.parametrize("dtype", ["bf16", "fp16"])
@pytest.mark.parametrize("S", CROSS_S)
@pytest.mark.parametrize("G", [1, 2, 3, 4, 5, 6, 7, 8])
@pytest.mark.parametrize("impl", [1, 2], ids=["split", "stream"])
def test_cross_attn_op(cuda, impl, G, S, dtype):
    """A in {1, 3, 16} x fp32 / 16-bit output x q final / 3 raw partial sums; needle and rising scores at A = 3; the alignment capture
    (NaN-filled buffer, head slots given out of order with -1 between) at steps inside and outside [0, Tcap); two launches on the
    same scratch give bit-identical outputs and leave the counters at zero."""
    g = torch.Generator(device="cpu").manual_seed(impl * 100000 + G * 10000 + S)
    H, D = CH, CH * 64
    slots = torch.tensor(HEAD_SLOTS, dtype=torch.int32, device=cuda)
    for A in (1, 3, 16):
        for mode in (("random", "needle", "rising") if A == 3 else ("random",)):
            q, kc, vc, needles = _cross_case(A, G, S, mode, g, cuda, dtype)
            vmax = vc.float().abs().max().item()
            scratch = _XScratch(A, G, H, cuda)
            for out_f32, nsplit in ((True, 0), (False, 3), (True, 3), (False, 0)):
                qin, bias, alpha, qeff = _q_input(q, nsplit, g, cuda)
                ref, sc = _ref_cross(qeff, kc, vc, A, G, H, S)
                step = [2, -1, TCAP, 0][(out_f32 + 2 * (nsplit > 0)) % 4]
                align = torch.full((A * G, HA, TCAP, S), float("nan"), device=cuda)
                rc, out = _cross_attn(qin, nsplit, bias, alpha, kc, vc, A, G, H, S, dtype, out_f32, impl, scratch, align, slots,
                                      STEP_BASE + step)
                _lib()[0].check(rc)
                torch.cuda.synchronize()
                tag = f"cross_attn {['', 'split', 'stream'][impl]} {dtype}"
                if mode == "needle":
                    want = torch.stack([vc[a, :, needles[a][g_]].reshape(D) for a in range(A) for g_ in range(G)]).double()
                    err = _out_err(out, want, vmax, dtype)
                    _note(f"{tag} needle", err, NEEDLE_BOUND)
                    assert err <= NEEDLE_BOUND, (A, needles, out_f32, nsplit, err)
                else:
                    err = _out_err(out, ref, vmax, dtype)
                    _note(f"{tag} {'fp32' if out_f32 else '16-bit'} out", err, CROSS_BOUND)
                    assert err <= CROSS_BOUND, (A, mode, out_f32, nsplit, err)
                assert (scratch.counters == 0).all(), "counters must be zero on return"
                # ---- alignment capture: row ((a*G + g)*Ha + slot)*Tcap + step, raw score of every key; nothing else written
                want = torch.full_like(align, float("nan"), dtype=torch.float64)
                if 0 <= step < TCAP:
                    for h, sl in enumerate(HEAD_SLOTS):
                        if sl >= 0:
                            want.view(A, G, HA, TCAP, S)[:, :, sl, step] = sc[:, :, h]
                written = ~torch.isnan(align)
                assert torch.equal(written, ~torch.isnan(want)), ("capture wrote the wrong rows", step)
                if written.any():
                    qn = qeff.view(A, G, H, 64).norm(dim=-1)  # [A, G, H]
                    kn = kc.double().norm(dim=-1)  # [A, H, S]
                    scale = torch.zeros_like(want)
                    for h, sl in enumerate(HEAD_SLOTS):
                        if sl >= 0:
                            scale.view(A, G, HA, TCAP, S)[:, :, sl, step] = qn[:, :, h, None] * kn[:, None, h]
                    aerr = ((align.double() - want).abs()[written] / scale[written].clamp_min(1e-30)).max().item()
                    _note(f"{tag} align score / (|q||k|)", aerr, ALIGN_BOUND)
                    assert aerr <= ALIGN_BOUND, (A, mode, step, aerr)
            # determinism: the same launch twice on the same scratch
            qin, bias, alpha, _ = _q_input(q, 3, g, cuda)
            rc1, o1 = _cross_attn(qin, 3, bias, alpha, kc, vc, A, G, H, S, dtype, True, impl, scratch)
            rc2, o2 = _cross_attn(qin, 3, bias, alpha, kc, vc, A, G, H, S, dtype, True, impl, scratch)
            assert rc1 == 0 and rc2 == 0
            torch.cuda.synchronize()
            assert torch.equal(o1, o2), "two launches differ"
            assert (scratch.counters == 0).all()


@pytest.mark.parametrize("impl", [0, 1, 2])
def test_cross_attn_rejects_before_launch(cuda, impl):
    """S > 1536 and G > 8 are refused by the host-side check: the BW_CHECK error code, and the output is not touched."""
    L, lib = _lib()
    for A, G, S in ((1, 1, MAXS + 1), (1, 9, 64), (2, 0, 64)):
        kc = torch.zeros(A, CH, S, 64, dtype=torch.bfloat16, device=cuda)
        scratch = _XScratch(A, max(G, 1), CH, cuda)
        q = torch.zeros(A * max(G, 1), CH * 64, device=cuda)
        rc, out = _cross_attn(q, 0, None, 1.0, kc, kc, A, G, CH, S, "bf16", True, impl, scratch)
        torch.cuda.synchronize()
        assert rc == BW_CHECK_RC, (A, G, S, rc)
        assert lib.bw_last_error()
        assert torch.isnan(out).all(), "a refused call wrote its output"


def test_cross_attn_policy_picks_by_cta_count(cuda, monkeypatch):
    """impl 0 = the engine's policy: the streaming kernel from BW_XATTN_STREAM_MIN CTAs (A * H) on.  The two kernels sum in different
    orders, so the result tells which one ran: below the threshold it is bit-identical to impl 1, from it on to impl 2."""
    g = torch.Generator(device="cpu").manual_seed(5)
    A, G, S = 2, 3, 500
    q, kc, vc, _ = _cross_case(A, G, S, "random", g, cuda, "bf16")
    outs = {}
    for impl in (1, 2):
        rc, outs[impl] = _cross_attn(q, 0, None, 1.0, kc, vc, A, G, CH, S, "bf16", True, impl, _XScratch(A, G, CH, cuda))
        assert rc == 0
    torch.cuda.synchronize()
    assert not torch.equal(outs[1], outs[2])
    for thr, want in ((A * CH + 1, 1), (A * CH, 2), (0, 1)):
        monkeypatch.setenv("BW_XATTN_STREAM_MIN", str(thr))
        rc, o = _cross_attn(q, 0, None, 1.0, kc, vc, A, G, CH, S, "bf16", True, 0, _XScratch(A, G, CH, cuda))
        assert rc == 0
        torch.cuda.synchronize()
        assert torch.equal(o, outs[want]), (thr, want)


# ------------------------------------------------------------------------------------------------------------------
# e. which step path ran
# ------------------------------------------------------------------------------------------------------------------
def step_path(eng, launches_before, n_steps):
    """'mega' / 'perop' / 'batched' from the kernels one decode_run step launched (bw_decode_kernel_launches, counted from the
    captured step graph): the persistent kernel is one launch (+ the select kernel without fused selection); the per-op step is the
    embedding, 8 per layer (QKV / out / q / xo / fc1 / fc2 GEMVs, self- and cross-attention), the LM head and the select kernel; the
    batched step is the embedding, 12 per layer (4 residual+LayerNorm ... ), the final LayerNorm, the LM head and the select kernel."""
    per = (eng.decode_kernel_launches() - launches_before) / n_steps
    L = eng.dims.dec_layers
    if per in (1, 2):
        return "mega"
    if per == 8 * L + 3:
        return "perop"
    if per == 12 * L + 4:
        return "batched"
    raise AssertionError(f"{per} kernels per step match no decoder step path (L = {L})")


PATH_ENV = {
    "mega": {"BW_NO_MEGA": "0", "BW_BATCH_MIN": "1000"},
    "perop": {"BW_NO_MEGA": "1", "BW_BATCH_MIN": "1000", "BW_XATTN_STREAM_MIN": "0"},
    "batched": {"BW_NO_MEGA": "1", "BW_BATCH_MIN": "1", "BW_XATTN_STREAM_MIN": "0"},
    "batched-xstream": {"BW_NO_MEGA": "1", "BW_BATCH_MIN": "1", "BW_XATTN_STREAM_MIN": "1"},
}


def _set_path(monkeypatch, path):
    for k in ("BW_NO_MEGA", "BW_BATCH_MIN", "BW_XATTN_STREAM_MIN"):
        monkeypatch.delenv(k, raising=False)
    for k, v in PATH_ENV[path].items():
        monkeypatch.setenv(k, v)
    return path.split("-")[0]


# ------------------------------------------------------------------------------------------------------------------
# c. long decode through the engine: all 448 positions, every step path
# ------------------------------------------------------------------------------------------------------------------
SEEDS = (1000, 1001)
BANDS = ((0, 128, "<128"), (128, 144, "128-143"), (144, 448, "144-447"))
# teacher-forced bounds in units of the logit sigma of the golden fixture: the bounds of test_model_gpu (tiny10) / test_large_gpu
# (turbo10) for the 16..36 positions they decode.  turbo10 bf16: 0.40, the bound test_large_gpu derives from HF's own bf16 path
# (1.5 x 0.25 sigma); measured on a B200 over 448 positions: 0.26 sigma below position 128 on every path, 0.31 at most above.
TF_SIGMA = {("tiny10", "bf16"): 0.08, ("tiny10", "fp16"): 0.02, ("turbo10", "bf16"): 0.40, ("turbo10", "fp16"): 0.30}
BAND_RATIO = 1.5
# admissible near ties per generated token (each one checked against the measured logit error): at turbo dims in bf16 the logit error
# is 0.26 sigma, and 12-14 % of 444 greedy steps have an oracle gap inside twice that (measured); 1-2 % elsewhere
NEAR_TIE_FRACTION = {("turbo10", "bf16"): 0.20}


class _Model:
    def __init__(self, tag):
        from oracle import hf_ref
        from thewhisper_b200 import synthetic as S

        meta = json.load(open(os.path.join(GOLD, f"model_{tag}.json")))
        self.tag, self.chunk = tag, meta["chunk_s"]
        self.gold = np.load(os.path.join(GOLD, f"model_{tag}.npz"))
        self.sigma = float(self.gold["tf_cols"].std())
        self.model = S.make_hf_model(meta["preset"], seed=meta["seed"], layer_gain=meta.get("layer_gain", 1.0))
        hf_ref.interpolate_positions(self.model, self.chunk)
        fe = S.make_feature_extractor(self.chunk)
        self.mels = {s: hf_ref.logmel(fe, S.synth_audio(self.chunk, seed=s)) for s in SEEDS}
        self.weights = {}
        self._enc = {}
        self._tf = {}

    def engine(self, Q, dtype, **kw):
        """a fresh engine (the step-path switches are read when it is created); the packed weights are kept per dtype"""
        from thewhisper_b200.engine import ModelDims, WhisperEngine

        et = E16[dtype][0]
        e = WhisperEngine(self.model.state_dict(), ModelDims.from_hf_config(self.model.config), chunk_length_s=self.chunk,
                          max_audios=Q, weights=self.weights.get(et), dtype=et, **kw)
        self.weights = {et: e.weights}
        return e

    def enc(self, seed):
        if seed not in self._enc:
            with torch.no_grad():
                self._enc[seed] = self.model.model.encoder(torch.from_numpy(self.mels[seed])[None]).last_hidden_state
        return self._enc[seed]

    def oracle_tf(self, seed, ids):
        key = (seed, tuple(ids))
        if key not in self._tf:
            with torch.no_grad():
                out = self.model(encoder_outputs=(self.enc(seed),), decoder_input_ids=torch.tensor([list(ids)], dtype=torch.long))
            self._tf[key] = out.logits[0].float().numpy()
        return self._tf[key]


_MODELS = {}


def _model(tag):
    if tag not in _MODELS:
        _MODELS.clear()
        _MODELS[tag] = _Model(tag)
    return _MODELS[tag]


def _opts(model, extra_suppress=(), align=False):
    from thewhisper_b200 import synthetic as S
    from thewhisper_b200.engine import DecodeOptions

    g = model.generation_config
    return DecodeOptions(eos_token=S.EOS, pad_token=S.EOS, suppress_tokens=list(g.suppress_tokens) + list(extra_suppress),
                         begin_suppress_tokens=list(g.begin_suppress_tokens), record_alignment=align)


LONG_CASES = [(p, q) for p, q in (("mega", 1), ("mega", 2), ("perop", 1), ("batched", 3), ("batched-xstream", 3))]


@pytest.mark.parametrize("dtype", ["bf16", "fp16"])
@pytest.mark.parametrize("path,Q", LONG_CASES, ids=[f"{p}-Q{q}" for p, q in LONG_CASES])
@pytest.mark.parametrize("tag", ["tiny10", "turbo10"])
def test_long_decode_every_path(cuda, tag, path, Q, dtype, monkeypatch):
    """Teacher-forced over all 448 positions (4-token prompt + 444 seeded text tokens, one prompt): logits of every position within
    the sigma bound of the short-decode tests, and the worst error at positions >= 128 (second key chunk of the self-attention
    kernel) and >= 144 (wide exp lanes of the persistent kernel) no worse than BAND_RATIO x the worst below 128.  Then greedy with
    EOS suppressed to the end of the cache: exactly 444 tokens, nothing written past Tmax, every token the oracle's arg-max unless
    the oracle's own gap is within twice the measured top-8 logit error."""
    from thewhisper_b200 import synthetic as S

    want_path = _set_path(monkeypatch, path)
    m = _model(tag)
    Tmax = m.model.config.max_target_positions
    assert Tmax == 448
    eng = m.engine(Q + 1, dtype)  # row Q: a guard row no decode touches
    seeds = [SEEDS[q % len(SEEDS)] for q in range(Q)]
    eng.set_mel(torch.from_numpy(np.stack([m.mels[s] for s in seeds])))
    eng.encode(Q)
    rng = np.random.RandomState(448)
    prompt = [S.SOT, S.LANG_EN, S.TRANSCRIBE, S.NOTIMESTAMPS]
    ids = np.array(prompt + rng.randint(0, S.EOS, size=Tmax - len(prompt)).tolist(), dtype=np.int32)
    refs = {s: m.oracle_tf(s, ids.tolist()) for s in sorted(set(seeds))}
    opts = _opts(m.model, extra_suppress=[S.EOS])
    # ---- teacher-forced, every position
    eng.decode_begin(np.tile(ids[None, :], (Q, 1)), Q, 1, opts)
    l0 = eng.decode_kernel_launches()
    per_pos = np.zeros(Tmax)
    worst_top = 0.0
    for t in range(Tmax):
        eng.decode_run(1)
        lg = eng.logits().cpu().numpy()
        for q in range(Q):
            if q >= len(SEEDS):
                assert np.array_equal(lg[q], lg[q % len(SEEDS)]), (t, q)  # same audio, same prefix: bit for bit
                continue
            ref = refs[seeds[q]][t]
            per_pos[t] = max(per_pos[t], float(np.abs(lg[q] - ref).max()))
            top = np.argpartition(-ref, 8)[:8]
            worst_top = max(worst_top, float(np.abs(lg[q][top] - ref[top]).max()))
    assert step_path(eng, l0, Tmax) == want_path
    bands = {name: per_pos[a:b].max() / m.sigma for a, b, name in BANDS}
    bound = TF_SIGMA[(tag, dtype)]
    print(f"\n[{tag} {path} Q={Q} {dtype}] teacher-forced max |dlogit| / sigma by position band: "
          + ", ".join(f"{k} {v:.4f}" for k, v in bands.items()) + f" (bound {bound}, bands >= 128 <= {BAND_RATIO} x band < 128)")
    assert max(bands.values()) < bound + 1e-3 / m.sigma, bands
    for name in ("128-143", "144-447"):
        assert bands[name] <= BAND_RATIO * bands["<128"], (name, bands)
    # ---- greedy to the end of the cache
    tok_rows = eng.max_audios * eng.max_beams
    before = eng.buffer("tokens", torch.int32, (tok_rows, Tmax)).cpu().numpy()
    gprompt = np.array([prompt] * Q, dtype=np.int32)
    l0 = eng.decode_kernel_launches()
    gen, toks, n = eng.greedy(gprompt, Q, opts, max_new_tokens=Tmax - len(prompt))
    assert step_path(eng, l0, Tmax - 1) == want_path
    assert n == Tmax - len(prompt)
    _, _, pos = eng.decode_read()
    assert pos == Tmax - 1, pos
    after = eng.buffer("tokens", torch.int32, (tok_rows, Tmax)).cpu().numpy()
    assert np.array_equal(after[Q:], before[Q:]), "tokens written past the last row's Tmax"
    assert (after[:Q, : len(prompt)] == np.array(prompt)[None, :]).all(), "a prompt was overwritten"
    tol = 2.0 * worst_top
    g = m.model.generation_config
    near = 0
    for q in range(min(Q, len(SEEDS))):
        assert len(gen[q]) == Tmax - len(prompt), len(gen[q])
        assert np.array_equal(after[q, len(prompt):], gen[q])
        ref_lg = m.oracle_tf(seeds[q], prompt + gen[q].tolist())
        for i, tok in enumerate(gen[q]):
            row = ref_lg[len(prompt) - 1 + i].copy()
            row[list(g.suppress_tokens) + [S.EOS]] = -np.inf
            if i == 0:
                row[list(g.begin_suppress_tokens)] = -np.inf
            best = int(np.argmax(row))
            if tok != best:
                gap = float(row[best] - row[tok])
                assert gap < tol, (q, i, int(tok), best, gap, tol)
                near += 1
    for q in range(len(SEEDS), Q):
        assert gen[q].tolist() == gen[q % len(SEEDS)].tolist(), q
    print(f"[{tag} {path} Q={Q} {dtype}] greedy: {Tmax - len(prompt)} tokens per row, {near} near ties (oracle gap < {tol:.4f})")
    assert near <= NEAR_TIE_FRACTION.get((tag, dtype), 0.05) * (Tmax - len(prompt)) * min(Q, len(SEEDS)), near
    eng.close()


# ------------------------------------------------------------------------------------------------------------------
# d. alignment scores recorded by the decoder step against the model's cross-attention
# ------------------------------------------------------------------------------------------------------------------
ALIGN_CASES = [("mega", 1, 1), ("perop", 1, 1), ("batched-xstream", 3, 1), ("beam-xstream", 2, 5)]
ALIGN_PROB_BOUND = 0.05  # max |softmax(engine scores) - HF cross-attention| of one key (probabilities); measured 0.0163
N_ALIGN = 32


@pytest.mark.parametrize("path,A,G", ALIGN_CASES, ids=[c[0] for c in ALIGN_CASES])
def test_alignment_capture_matches_cross_attention(cuda, path, A, G, monkeypatch):
    """Greedy (EOS suppressed) with record_alignment for 33 steps: the 32 rows recorded per sequence slot, softmaxed over S, must match
    HF's eager cross-attention of the alignment heads for the same prefix, and the word-timestamp pass over them must give the jump
    times of whisper_ref.token_timestamps on HF's attention (within the tolerance of test_word_timestamps_kernels' noisy case).
    beam-xstream: A = 2 audios x G = 5 beams on cross_attn_stream_kernel<5>; beam g takes its g-th candidate at the first step and
    its best one after that, so the five slots of an audio hold five different sequences."""
    from oracle import whisper_ref
    from thewhisper_b200 import synthetic as S
    from thewhisper_b200.engine import ModelDims, WhisperEngine

    want_path = _set_path(monkeypatch, "batched-xstream" if path == "beam-xstream" else path)
    m = _model("tiny10")
    heads = [list(map(int, p)) for p in m.model.generation_config.alignment_heads]
    Ha, Q = len(heads), A * G
    eng = WhisperEngine(m.model.state_dict(), ModelDims.from_hf_config(m.model.config), chunk_length_s=m.chunk, max_audios=A,
                        max_beams=G, alignment_heads=heads, max_align_steps=64)
    seeds = [SEEDS[a % len(SEEDS)] for a in range(A)]
    eng.set_mel(torch.from_numpy(np.stack([m.mels[s] for s in seeds])))
    eng.encode(A)
    Sk, Tcap = eng.S, eng.max_align_steps
    prompt = [S.SOT, S.LANG_EN, S.TRANSCRIBE, S.NOTIMESTAMPS]
    opts = _opts(m.model, extra_suppress=[S.EOS], align=True)
    eng.write_buffer("align", torch.full((Q * Ha * Tcap * Sk,), float("nan"), device=cuda))
    l0 = eng.decode_kernel_launches()
    if G == 1:
        gen, _, _ = eng.greedy(np.array([prompt] * Q, dtype=np.int32), A, opts, max_new_tokens=N_ALIGN + 1)
        seqs = [prompt + gen[q].tolist() for q in range(Q)]
        n_steps = len(prompt) - 1 + N_ALIGN + 1
    else:
        eng.decode_begin(np.array([prompt] * Q, dtype=np.int32), A, G, opts)
        eng.decode_run(len(prompt) - 1)
        seqs = [list(prompt) for _ in range(Q)]
        for step in range(N_ALIGN + 1):
            _, ct = eng.decode_beam_step(np.zeros(Q, dtype=np.float32))
            if step == N_ALIGN:
                break
            nxt = np.array([ct[q][ct[q] >= 0][q % G if step == 0 else 0] for q in range(Q)], dtype=np.int32)
            eng.decode_reorder(np.arange(Q, dtype=np.int32), nxt)
            for q in range(Q):
                seqs[q].append(int(nxt[q]))
        for a in range(A):
            assert len({tuple(s) for s in seqs[a * G:(a + 1) * G]}) == G, "the beams of an audio must hold different sequences"
        n_steps = len(prompt) - 1 + N_ALIGN + 1
    assert step_path(eng, l0, n_steps) == want_path
    align = eng.buffer("align", torch.float32, (Q, Ha, Tcap, Sk)).cpu()
    # row t: the step whose input is position begin_index + t; rows past the decoded steps stay untouched
    assert not torch.isnan(align[:, :, :N_ALIGN]).any(), "a recorded row holds NaN"
    assert torch.isnan(align[:, :, N_ALIGN:]).all(), "rows past the decoded steps were written"
    got = torch.softmax(align[:, :, :N_ALIGN].double(), dim=-1).numpy()  # [Q, Ha, T, S]
    m.model.config._attn_implementation = "eager"
    worst, bad, total, devs = 0.0, 0, 0, []
    mine_all = np.concatenate([eng.word_timestamps_batch(list(range(q0, min(q0 + A, Q))), [N_ALIGN] * min(A, Q - q0), [Sk] * min(A, Q - q0))
                               for q0 in range(0, Q, A)])  # (at most max_audios slots per call)
    for q in range(Q):
        ids = torch.tensor([seqs[q][: len(prompt) + N_ALIGN]], dtype=torch.long)
        with torch.no_grad():
            out = m.model.model.decoder(input_ids=ids, encoder_hidden_states=m.enc(seeds[q // G]), output_attentions=True)
        ref = np.stack([out.cross_attentions[l][0, h, len(prompt):len(prompt) + N_ALIGN].float().numpy() for l, h in heads])
        worst = max(worst, float(np.abs(got[q] - ref).max()))
        with np.errstate(all="ignore"):
            want_ts = whisper_ref.token_timestamps(ref.astype(np.float32), Sk, 0.02)
        mine = mine_all[q, : N_ALIGN + 1]
        same = (mine == want_ts) | (np.isnan(mine) & np.isnan(want_ts))
        bad += int((~same).sum())
        total += len(want_ts)
        devs += np.abs(np.nan_to_num(mine) - np.nan_to_num(want_ts)).tolist()
    print(f"\n[alignment {path} A={A} G={G}] max |softmax(scores) - HF cross-attention| = {worst:.5f} (bound {ALIGN_PROB_BOUND}); "
          f"{bad} of {total} jump times differ, median |d| {np.median(devs):.3f} s (bounds {0.45 * total:.0f}, 0.02 s)")
    assert worst <= ALIGN_PROB_BOUND, worst
    assert bad <= 0.45 * total and np.median(devs) <= 0.0200001, (bad, total, np.median(devs))
    eng.close()
