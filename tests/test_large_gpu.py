"""Parity at the dimensions that are benchmarked (VERDICT round 1, missing #1): BASELINE.json configs C1 (whisper-large-v3-turbo
dims, 10 s chunk) and C2 (whisper-large-v3 dims, 30 s chunk) against

  * the golden fixtures minted from the REAL reference in the build container (tests/golden/model_turbo10.*, model_large30.*,
    `oracle/make_golden.py --large`: fp32 HF path of REF thestage_speechkit/nvidia/asr_pipeline.py:30-92), and
  * the oracle run live on this box's host cores (oracle/hf_ref.py) for the rows / prefixes the fixtures do not hold.

What runs at these dimensions and nowhere else in the suite: `decode_mega_kernel` with R = 3 weight slabs per warp, the
double-buffered slab plan and 7 cross-attention key splits (Q = 1 and Q = 2); the batched step at Q = 3 / 8 / 64; the encoder at
S = 1500 (12 query tiles, ragged last key tile) through 32 layers.

Protocol (SURVEY.md section 7 hard part 1): teacher-forced logits at every position within a stated fraction of the logit standard
deviation; free-running greedy ids must equal the oracle's processed arg-max given the same prefix at every step whose oracle
top-1/top-2 margin exceeds twice the measured logit error -- the admissible near ties are counted, bounded and printed.
The checkpoints are random (no weights offline) with layer_gain 4 so that sequences depend on the audio."""
import json
import os

import numpy as np
import pytest
import torch

from tests.conftest import GOLD

pytestmark = pytest.mark.gpu

# Measured on the B200 (profiles/r2_parity_large.md, gpurun r2a): max |dlogit| over 16 teacher-forced positions = 0.11-0.12 sigma on the
# golden sub-sample of audio 1000 and 0.19-0.20 sigma over the FULL 51866-column rows of the other audios (same number for the
# persistent kernel, the per-op kernels and the batched path: the error is the bf16 operand rounding of 32 encoder + 4/32 decoder
# layers with gain-4 weights, not a property of one kernel); encoder output mean |err| 0.019-0.027 on a unit-scale LayerNorm
# output.  The test also measures how far HF's own bf16 CUDA path is from the fp32 oracle on the same box (printed beside ours):
# the bound is the larger of 1.5 x that and the absolute cap below.
LOGIT_CAP_SIGMA = 0.30
ENC_TOL = {"turbo10": (0.30, 0.045), "large30": (0.30, 0.035)}  # (max abs, mean abs) of the final-LayerNorm output (unit scale)
SEEDS = (1000, 1001, 1002, 1003)
# step-path switches an engine reads once, when it is created: part of the engine cache key, so a test that sets one gets a fresh engine
PATH_SWITCHES = ("BW_NO_MEGA", "BW_BATCH_MIN", "BW_XATTN_STREAM_MIN")


class Case:
    def __init__(self, tag):
        from oracle import hf_ref
        from thewhisper_b200 import synthetic as S

        self.tag = tag
        self.meta = json.load(open(os.path.join(GOLD, f"model_{tag}.json")))
        self.gold = np.load(os.path.join(GOLD, f"model_{tag}.npz"))
        self.chunk = self.meta["chunk_s"]
        self.model = S.make_hf_model(self.meta["preset"], seed=self.meta["seed"], layer_gain=self.meta["layer_gain"])
        if self.chunk < 30:
            hf_ref.interpolate_positions(self.model, self.chunk)  # the oracle's copy of REF patch_hf_model
        fe = S.make_feature_extractor(self.chunk)
        self.mels = {s: hf_ref.logmel(fe, S.synth_audio(self.chunk, seed=s)) for s in SEEDS}
        self._engines = {}
        self._weights = {}
        self._tf = {}
        self._enc = {}

    def engine(self, max_audios, dtype=torch.bfloat16):
        from thewhisper_b200.engine import ModelDims, WhisperEngine

        key = (max_audios, dtype, tuple(os.environ.get(k) for k in PATH_SWITCHES))
        for k in list(self._engines):  # one engine alive at a time (cross K/V of 64 audios = 15.7 GB)
            if k != key:
                self._engines.pop(k).close()
        if key not in self._engines:
            e = WhisperEngine(self.model.state_dict(), ModelDims.from_hf_config(self.model.config), chunk_length_s=self.chunk,
                              max_audios=max_audios, weights=self._weights.get(dtype), dtype=dtype)
            self._weights = {dtype: e.weights}  # (one packed copy alive at a time)
            self._engines[key] = e
        return self._engines[key]

    def hf_bf16_err(self, seed, ids):
        """max |logit(HF bf16 on this GPU) - logit(fp32 oracle)| over the same teacher-forced sequence: the noise floor of the
        reference's own reduced-precision path (SURVEY.md section 7 hard part 1a), measured, not assumed."""
        key = ("hf", seed, tuple(ids))
        if key not in self._tf:
            import copy

            m = copy.deepcopy(self.model).to(device="cuda", dtype=torch.bfloat16)
            with torch.no_grad():
                out = m(input_features=torch.from_numpy(self.mels[seed])[None].to("cuda", torch.bfloat16),
                        decoder_input_ids=torch.tensor([list(ids)], dtype=torch.long, device="cuda"))
            lg = out.logits[0].float().cpu().numpy()
            del m, out
            torch.cuda.empty_cache()
            self._tf[key] = float(np.abs(lg - self.oracle_tf(seed, ids)).max())
        return self._tf[key]

    def oracle_tf(self, seed, ids):
        """Live oracle logits [T, V] for a token sequence over audio `seed` (cached per call signature)."""
        from oracle import hf_ref

        key = (seed, tuple(ids))
        if key not in self._tf:
            if seed not in self._enc:  # the encoder pass of an audio is run once, not once per token sequence
                with torch.no_grad():
                    self._enc[seed] = self.model.model.encoder(torch.from_numpy(self.mels[seed])[None]).last_hidden_state
            with torch.no_grad():
                out = self.model(encoder_outputs=(self._enc[seed],), decoder_input_ids=torch.tensor([list(ids)], dtype=torch.long))
            self._tf[key] = out.logits[0].float().numpy()
        return self._tf[key]


_CASES = {}


@pytest.fixture(scope="module")
def case(request):
    tag = request.param
    if tag not in _CASES:
        _CASES.clear()  # drop the other size's model + engine before building this one
        _CASES[tag] = Case(tag)
    return _CASES[tag]


def _opts(model):
    from thewhisper_b200 import synthetic as S
    from thewhisper_b200.engine import DecodeOptions

    g = model.generation_config
    return DecodeOptions(eos_token=S.EOS, pad_token=S.EOS, suppress_tokens=list(g.suppress_tokens),
                         begin_suppress_tokens=list(g.begin_suppress_tokens))


@pytest.mark.parametrize("case", ["turbo10", "large30"], indirect=True)
def test_encoder_at_benchmark_dims(cuda, case):
    """32 encoder layers at S = 500 / 1500 against the reference's own encoder output (golden sub-sample, fp32) and the live oracle."""
    eng = case.engine(2)
    mels = np.stack([case.mels[1000], case.mels[1001]])
    eng.set_mel(torch.from_numpy(mels))
    eng.encode(2)
    out = eng.encoder_output(2).cpu().numpy()
    case.oracle_tf(1001, [50258])  # fills the oracle's encoder-output cache for audio 1001
    ref1 = case._enc[1001][0].float().numpy()
    sub = case.gold["enc_sub"]
    step_r, step_c = max(1, out.shape[1] // 50), max(1, out.shape[2] // 64)
    e0 = np.abs(out[0][::step_r, ::step_c] - sub)
    e1 = np.abs(out[1] - ref1)
    print(f"\n[{case.tag}] encoder |err| vs golden sub-sample: max {e0.max():.4f} mean {e0.mean():.5f}; "
          f"vs live oracle (audio 1001, all {out[1].size} values): max {e1.max():.4f} mean {e1.mean():.5f}")
    mx, mean = ENC_TOL[case.tag]
    assert e0.max() < mx and e0.mean() < mean, (e0.max(), e0.mean())
    assert e1.max() < mx and e1.mean() < mean, (e1.max(), e1.mean())


def _decode_check(case, Q, monkeypatch, env=None, dtype=torch.bfloat16, want_path=None):
    """Teacher-forced logits at every position + free-running greedy (tie-aware) for Q sequences over audios SEEDS[q % 4].
    want_path: the decoder step path ('mega' / 'perop' / 'batched') the teacher-forced steps must have run."""
    from tests.test_decoder_attn_gpu import step_path
    from thewhisper_b200 import synthetic as S

    for k, v in (env or {}).items():
        monkeypatch.setenv(k, v)
    gold, model = case.gold, case.model
    eng = case.engine(Q, dtype)
    seeds = [SEEDS[q % len(SEEDS)] for q in range(Q)]
    eng.set_mel(torch.from_numpy(np.stack([case.mels[s] for s in seeds])))
    eng.encode(Q)
    opts = _opts(model)
    ids = gold["tf_ids"].astype(np.int32)
    sigma = float(gold["tf_cols"].std())
    # ---- teacher-forced: every position, every row.  Rows over audio 1000 against the golden top-8 / strided columns minted from
    #      the real reference; rows over the other audios against the live oracle (full rows)
    eng.decode_begin(np.tile(ids[None, :], (Q, 1)), Q, 1, opts)
    worst, worst_top = 0.0, 0.0
    uniq = sorted(set(seeds))
    refs = {s: case.oracle_tf(s, ids.tolist()) for s in uniq if s != 1000}
    first_row = {s: seeds.index(s) for s in uniq}
    launches0 = eng.decode_kernel_launches()
    for t in range(len(ids)):
        eng.decode_run(1)
        lg = eng.logits().cpu().numpy()
        for q in range(Q):
            if q != first_row[seeds[q]]:
                assert np.array_equal(lg[q], lg[first_row[seeds[q]]]), (t, q)  # same audio + same prefix -> same logits, bit for bit
                continue
            if seeds[q] == 1000:
                worst = max(worst, float(np.abs(lg[q][::997] - gold["tf_cols"][t]).max()))
                top = gold["tf_top_ids"][t]
                worst_top = max(worst_top, float(np.abs(lg[q][top] - gold["tf_top_vals"][t]).max()))
            else:
                ref_row = refs[seeds[q]][t]
                worst = max(worst, float(np.abs(lg[q] - ref_row).max()))
                top = np.argsort(-ref_row)[:8]
                worst_top = max(worst_top, float(np.abs(lg[q][top] - ref_row[top]).max()))
    if want_path is not None:
        assert step_path(eng, launches0, len(ids)) == want_path
    worst = max(worst, worst_top)
    hf_err = case.hf_bf16_err(1001, ids.tolist())
    print(f"\n[{case.tag} Q={Q} {env or 'default'} {str(dtype).replace('torch.', '')}] teacher-forced max |dlogit| = {worst:.4f} = {worst / sigma:.4f} sigma (sigma {sigma:.3f}); "
          f"HF bf16 on this GPU vs the same fp32 oracle (audio 1001, full rows): {hf_err:.4f} = {hf_err / sigma:.4f} sigma")
    assert worst < max(LOGIT_CAP_SIGMA * sigma, 1.5 * hf_err), (worst, sigma, hf_err)
    # a greedy decision is a comparison of the two largest logits: its admissible margin is twice the error measured AT the top-8
    # logits of every row (smaller than the maximum over all 51866 columns printed above)
    tol = 2.0 * worst_top
    print(f"[{case.tag} Q={Q}] max |dlogit| at the oracle's top-8 tokens: {worst_top:.4f} -> near-tie margin {tol:.4f}")
    # ---- free-running greedy
    prompt = np.array([[S.SOT, S.LANG_EN, S.TRANSCRIBE, S.NOTIMESTAMPS]] * Q, dtype=np.int32)
    n_new = int(len(gold["greedy_tokens"]))
    gen, _, _ = eng.greedy(prompt, Q, opts, max_new_tokens=n_new)
    g = model.generation_config
    near = 0
    for q in range(Q):
        if q != first_row[seeds[q]]:
            assert gen[q].tolist() == gen[first_row[seeds[q]]].tolist(), q
            continue
        full = prompt[0].tolist() + gen[q].tolist()
        ref_lg = case.oracle_tf(seeds[q], full)
        row_near = 0
        for i, tok in enumerate(gen[q]):
            row = ref_lg[3 + i].copy()
            row[list(g.suppress_tokens)] = -np.inf
            if i == 0:
                row[list(g.begin_suppress_tokens)] = -np.inf
            order = np.argsort(-row)[:2]
            if tok != order[0]:
                # admissible iff the oracle itself rates the engine's token within the measured logit error of its own arg-max
                # (with 51866 columns several tokens can sit inside that band, not only the runner-up)
                gap = float(row[order[0]] - row[tok])
                assert gap < tol, (q, i, int(tok), order.tolist(), gap, tol)
                row_near += 1
        near += row_near
        if seeds[q] == 1000 and row_near == 0:  # golden greedy ids of the real reference
            gg = gold["greedy_tokens"]
            gg = gg[gg != S.EOS]
            assert gen[q].tolist() == gg[: len(gen[q])].tolist()
    print(f"[{case.tag} Q={Q}] greedy: {sum(len(x) for x in gen)} tokens, {near} admissible near ties (oracle margin < {tol:.4f})")
    assert near <= 4 * len(uniq), near  # measured: 2 per 32-token sequence at large-v3 dims
    return worst / sigma, near


@pytest.mark.parametrize("case", ["turbo10", "large30"], indirect=True)
@pytest.mark.parametrize("Q", [1, 2])
def test_decoder_mega_at_benchmark_dims(cuda, case, Q, monkeypatch):
    """The persistent one-kernel decoder step (the kernel bench.py times) at large-v3 / turbo dimensions."""
    _decode_check(case, Q, monkeypatch)


@pytest.mark.parametrize("case", ["turbo10", "large30"], indirect=True)
@pytest.mark.parametrize("Q", [3, 8, 64])
def test_decoder_batched_at_benchmark_dims(cuda, case, Q, monkeypatch):
    """The batched decoder step (what C3 / C4 / C5 run) at large-v3 / turbo dimensions."""
    _decode_check(case, Q, monkeypatch)


@pytest.mark.parametrize("case", ["large30"], indirect=True)
def test_decoder_perop_q1_at_benchmark_dims(cuda, case, monkeypatch):
    """The per-op kernels at Q = 1 (BW_NO_MEGA=1): what beams and the timestamp rules run."""
    _decode_check(case, 1, monkeypatch, env={"BW_NO_MEGA": "1"}, want_path="perop")


@pytest.mark.parametrize("case", ["large30"], indirect=True)
@pytest.mark.parametrize("Q", [1, 8])
def test_decoder_fp16_at_benchmark_dims(cuda, case, Q, monkeypatch):
    """The float16 build of the engine (bw_config::dtype = 1: what the reference's streaming / benchmark paths run) at large-v3
    dimensions, persistent kernel and batched step, against the same fp32 oracle: three more mantissa bits than bf16."""
    rel, near = _decode_check(case, Q, monkeypatch, dtype=torch.float16)
    assert rel < 0.10, rel  # (bf16 measures 0.11-0.19 sigma on the same checks)
