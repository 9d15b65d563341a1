#!/usr/bin/env python
"""cfg5 on the B200 (SURVEY.md 8d-5, row A10): on-device features feeding the reference's ConformerMutiLangModel.

B = 128 utterances of 8 s (seed 4, normalize_wav(randn)); random-init model (torch.manual_seed(0)), eval, lang=None
(ref: lid/ConformerLangModel.py:77-83, :272-294).  The model code is the UNMODIFIED reference, staged from
/root/reference into the git-ignored baseline/_ref/ by __graft_entry__.build() (the GPU box has no /root/reference).
  * consumer check: features from the fused kernel vs features from the oracle (CPU, the reference's arithmetic), both
    pushed through the same model on the GPU: CTC logits and language-id scores must agree;
  * timing: front-end + model forward per batch (CUDA events), end-to-end audio-s/s and the front-end's share.
Prints one JSON line.  usage: cfg5_device.py [B] [n_check]"""
import json, os, sys, types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
REF = os.path.join(ROOT, "baseline", "_ref")


def load_reference_model():
    if not os.path.exists(os.path.join(REF, "lid", "ConformerLangModel.py")):
        return None

    def stub(name, **attrs):
        m = types.ModuleType(name)
        for k, v in attrs.items():
            setattr(m, k, v)
        sys.modules[name] = m

    class _Metric:            # torchmetrics objects are only constructed by the model
        def __init__(self, *a, **k):
            pass

    try:
        import torchmetrics  # noqa: F401
    except Exception:
        stub("torchmetrics", WER=_Metric, CharErrorRate=_Metric, Accuracy=_Metric, WordErrorRate=_Metric)
    try:
        import torch.utils.tensorboard  # noqa: F401
    except Exception:
        stub("torch.utils.tensorboard", SummaryWriter=_Metric)
    sys.path.insert(0, REF)
    from lid.ConformerLangModel import ConformerMutiLangModel
    return ConformerMutiLangModel


def stand_in_model():
    """A consumer of the reference model's shape (SURVEY.md 3.5) built from torchaudio.models.Conformer, for the consumer
    check where the reference's model source is not staged: Conv1d subsampling (k=3, s=2, p=1), 14 Conformer blocks,
    one CTC head per language (vocab + blank) and a language-id head on the time-averaged encoding.  Not the reference
    model: it checks that the kernel's features drive a Conformer like the oracle's (the reference's arithmetic) do."""
    import torch
    from torchaudio.models import Conformer

    class StandInConformerLid(torch.nn.Module):
        def __init__(self, lang2vocab, lang2index, dim=176, **_):
            super().__init__()
            self.sub = torch.nn.Conv1d(80, dim, 3, stride=2, padding=1)
            self.enc = Conformer(input_dim=dim, num_heads=4, ffn_dim=4 * dim, num_layers=14, depthwise_conv_kernel_size=31)
            self.ctc = torch.nn.ModuleDict({k: torch.nn.Linear(dim, v + 1) for k, v in lang2vocab.items()})
            self.lid = torch.nn.Linear(dim, len(lang2index))

        def forward(self, x, sample_rate, lang):
            h = self.sub(x.transpose(1, 2)).transpose(1, 2)
            h, _ = self.enc(h, torch.full((h.shape[0],), h.shape[1], device=h.device))
            return {k: head(h).log_softmax(-1) for k, head in self.ctc.items()}, self.lid(h.mean(1)).softmax(-1)

    return StandInConformerLid


def run(B=128, n_check=16, steps=5, model=None):
    """model: the consumer's class; default the staged reference model (None is returned when it is not staged)."""
    import torch
    import speech_lid_b200 as lid
    from oracle import frontend_oracle as O
    Model = model or load_reference_model()
    if Model is None:
        return None
    dev = torch.device("cuda:0")
    N = 128000
    g = torch.Generator().manual_seed(4)
    wavs = [O.normalize_wav(torch.randn(1, N, generator=g)) for _ in range(B)]
    torch.manual_seed(0)
    model = Model(lang2vocab={"Persian": 40, "Swahili": 30, "Vietnamese": 90},
                  lang2index={"Persian": 0, "Swahili": 1, "Vietnamese": 2}, conformer_linear=True, sub_sampling=2).eval().to(dev)
    fe = lid.FrontEnd(n_mels=80)
    plan = fe.make_plan([N] * B, padded=True)
    packed = fe.pack([w.to(dev) for w in wavs], plan)
    feats = torch.empty(B, plan.t_max, 80, device=dev)

    def flat(out, lid_out):
        t = []
        for k in sorted(out.keys()):
            t.append(("ctc[%s]" % k, out[k]))
        lo = lid_out[0] if isinstance(lid_out, (list, tuple)) else lid_out
        if torch.is_tensor(lo):
            t.append(("lid", lo))
        return t

    # ---- consumer check on the first n_check utterances: device features vs oracle features through the same model
    n_check = min(n_check, B)
    fe.featurize_packed(packed, plan, out=feats)
    ours = feats[:n_check].clone()
    ref = torch.stack([O.kaldi_fbank(w) for w in wavs[:n_check]]).to(dev)
    with torch.no_grad():
        o1, l1 = model(ours, 16000, None)
        o2, l2 = model(ref, 16000, None)
    worst, agree = 0.0, 1.0
    detail = {}
    for (k, a), (_, b) in zip(flat(o1, l1), flat(o2, l2)):
        e = float((a - b).abs().max())
        ag = float((a.argmax(-1) == b.argmax(-1)).float().mean())
        detail[k] = dict(max_abs_diff=e, ref_abs_max=float(b.abs().max()), argmax_agreement=ag)
        worst, agree = max(worst, e), min(agree, ag)
    feat_err = float((ours - ref).abs().max() / ref.abs().max())

    # ---- timing: front-end + forward, whole batch
    def step():
        fe.featurize_packed(packed, plan, out=feats)
        with torch.no_grad():
            return model(feats, 16000, None)

    for _ in range(2):
        step()
    torch.cuda.synchronize()
    e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    fe_ms = tot_ms = 0.0
    for _ in range(steps):
        e[0].record()
        fe.featurize_packed(packed, plan, out=feats)
        e[1].record()
        with torch.no_grad():
            model(feats, 16000, None)
        e[2].record()
        torch.cuda.synchronize()
        fe_ms += e[0].elapsed_time(e[1])
        tot_ms += e[0].elapsed_time(e[2])
    fe_ms /= steps
    tot_ms /= steps
    audio_s = B * N / 16000.0
    consumer = "reference ConformerMutiLangModel" if model is None else Model.__name__
    return dict(workload="cfg5: %d x 8-s utterances -> fused fbank -> %s forward (random init, eval, fp32) on one B200" % (B, consumer),
                features_norm_rel_vs_oracle=feat_err, consumer_worst_abs_diff=worst, consumer_min_argmax_agreement=agree,
                checked_utterances=n_check, consumer=detail, ms_per_batch=round(tot_ms, 3), frontend_ms=round(fe_ms, 4),
                frontend_share=round(fe_ms / tot_ms, 5), e2e_audio_s_per_s=round(audio_s / (tot_ms * 1e-3), 1),
                frontend_audio_s_per_s=round(audio_s / (fe_ms * 1e-3), 1))


if __name__ == "__main__":
    B = int(sys.argv[1]) if len(sys.argv) > 1 else 128
    n_check = int(sys.argv[2]) if len(sys.argv) > 2 else 16
    r = run(B, n_check)
    print(json.dumps(r if r is not None else {"unavailable": "baseline/_ref/lid is missing (run __graft_entry__.build() where /root/reference exists)"}))
