"""CPU tier: host-side mirror of the reference surface, C-ABI export check, no-GPU behaviour."""
import ctypes
import json
import os
import re
import sys
import types

import pytest
import torch

import sovits_b200
from sovits_b200 import lib as L
from sovits_b200 import models, synth
from sovits_b200.frontend import f0_to_coarse
import svc_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _model_kwargs():
    with open(sovits_b200.DEFAULT_CONFIG) as f:
        return json.load(f)["model"]


def test_library_exports_every_declared_symbol():
    """The C-ABI library loads (no compute call) and exports every function include/sovits_b200.h declares."""
    header = open(os.path.join(ROOT, "include", "sovits_b200.h")).read()
    declared = set(re.findall(r"SVB_API\s+[\w\s\*]+?\b(svb_\w+)\s*\(", header))
    assert declared, "no declarations parsed"
    assert declared == set(L.SIGNATURES), declared ^ set(L.SIGNATURES)
    lib = L.load_library()
    for name in declared:
        assert hasattr(lib, name), name
    assert b"sm_100a" in lib.svb_version()
    assert lib.svb_strerror(-6) == b"unsupported configuration"


def test_state_dict_layout_matches_reference_keys(cfg, sd):
    net = models.SynthesizerTrn(1025, 20, **_model_kwargs())
    own = net.state_dict()
    assert set(own) == set(sd)
    for k, v in sd.items():
        assert tuple(own[k].shape) == tuple(v.shape), k
    # a reference checkpoint also carries enc_q.* / f0_decoder.*: they must be tolerated
    extra = dict(sd)
    extra["enc_q.pre.weight"] = torch.zeros(192, 1025, 1)
    net.load_state_dict(extra)
    assert torch.equal(net.state_dict()["dec.ups.0.weight_v"], sd["dec.ups.0.weight_v"])


def test_frontend_matches_oracle_prefix(cfg, sd):
    net = models.SynthesizerTrn(1025, 20, **_model_kwargs()).eval()
    net.load_state_dict(sd)
    c, f0, uv, sid = synth.golden_inputs(cfg, "b2_t24")
    noise = synth.draw_noise(2, 24, cfg)
    with torch.no_grad():
        x_mask = torch.ones(2, 1, 24)
        x = net.pre(c) * x_mask + net.emb_uv(uv.long()).transpose(1, 2)
        for flag in (True, False):
            z_p, _, _, _ = net.enc_p(x, x_mask, f0_to_coarse(f0), noice_scale=0.4, z_noise=noise["z_noise"], all_ones_mask=flag)
            xo, xm, _ = O.prologue(sd, c, f0, uv, sid, cfg, torch.float32)
            zo, _, _ = O.text_encoder(sd, xo, xm, O.f0_to_coarse(f0), noise["z_noise"], 0.4, cfg, torch.float32)
            assert torch.allclose(z_p, zo, atol=1e-5)


def test_infer_fails_loudly_without_cuda(cfg, sd):
    net = models.SynthesizerTrn(1025, 20, **_model_kwargs()).eval()
    net.load_state_dict(sd)
    c, f0, uv, sid = synth.golden_inputs(cfg, "b1_t33")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        net.infer(c, f0, uv, g=sid)


def test_unsupported_configs_are_rejected():
    kw = _model_kwargs()
    kw["use_depthwise_conv"] = True
    with pytest.raises(NotImplementedError):
        models.SynthesizerTrn(1025, 20, **kw)
    kw = _model_kwargs()
    kw["use_transformer_flow"] = True
    with pytest.raises(NotImplementedError):
        models.SynthesizerTrn(1025, 20, **kw)


def test_snake_variant_state_dict_layout(cfg):
    """vocoder_name='nsf-snake-hifigan' (BASELINE config 4) adds the SnakeAlias keys of hifiganwithsnake/models.py."""
    from sovits_b200.config import load_config
    cfg_s = load_config()
    cfg_s.vocoder_name = "nsf-snake-hifigan"
    kw = _model_kwargs()
    kw["vocoder_name"] = "nsf-snake-hifigan"
    net = models.SynthesizerTrn(1025, 20, **kw)
    sd_s = synth.synth_state_dict(cfg_s)
    assert set(net.state_dict()) == set(sd_s)
    assert "dec.resblocks.7.activations.5.act.beta" in sd_s and "dec.snake_post.downsample.lowpass.filter" in sd_s


def test_patch_reference_keeps_surface(cfg, sd, monkeypatch):
    """The zero-edit integration (INTEGRATION.md): ``patch_reference`` subclasses the reference's own SynthesizerTrn.  The
    reference's constructor / ``infer`` parameters and state_dict layout are stored in tests/golden/ref_surface.json
    (make_golden_surface.py); the patch is applied to a stand-in with that surface, whose ``enc_p`` takes the reference's
    call, and the patched prefix must reproduce the reference's own z_p."""
    import numpy as np
    from sovits_b200 import frontend
    with open(os.path.join(ROOT, "tests", "golden", "ref_surface.json")) as f:
        surface = json.load(f)
    code = models.SynthesizerTrn.__init__.__code__
    assert list(code.co_varnames[1:code.co_argcount]) == surface["init_params"]
    assert "vol" in surface["infer_params"] and "predict_f0" in surface["infer_params"]
    ref_layout = surface["state_dict"]
    assert all(ref_layout.get(k) == list(v.shape) for k, v in sd.items())
    assert all(k.startswith(("enc_q.", "f0_decoder.")) for k in set(ref_layout) - set(sd))

    class RefCallPriorEncoder(frontend.PriorEncoder):          # the reference's call: enc_p(x, x_mask, f0=..., noice_scale=...)
        def forward(self, x, x_mask, f0=None, noice_scale=1):
            return super().forward(x, x_mask, f0, noice_scale)

    class RefSynthesizerTrn(torch.nn.Module):
        """The reference class as patch_reference sees it: its constructor, the prefix modules infer calls, and every other
        parameter at the reference's key and shape."""

        def __init__(self, spec_channels, segment_size, inter_channels, hidden_channels, filter_channels, n_heads, n_layers,
                     kernel_size, p_dropout, resblock, resblock_kernel_sizes, resblock_dilation_sizes, upsample_rates,
                     upsample_initial_channel, upsample_kernel_sizes, gin_channels, ssl_dim, n_speakers, sampling_rate=44100,
                     vol_embedding=False, vocoder_name="nsf-hifigan", use_depthwise_conv=False, use_automatic_f0_prediction=True,
                     flow_share_parameter=False, n_flow_layer=4, n_layers_trans_flow=3, use_transformer_flow=False, **kwargs):
            super().__init__()
            self.vol_embedding, self.use_automatic_f0_prediction, self.character_mix = vol_embedding, use_automatic_f0_prediction, False
            self.emb_g = torch.nn.Embedding(n_speakers, gin_channels)
            self.pre = torch.nn.Conv1d(ssl_dim, hidden_channels, kernel_size=5, padding=2)
            self.enc_p = RefCallPriorEncoder(inter_channels, hidden_channels, filter_channels, n_heads, n_layers, kernel_size)
            self.emb_uv = torch.nn.Embedding(2, hidden_channels)
            for sub in ("flow", "dec", "enc_q", "f0_decoder"):
                setattr(self, sub, models._ParamTree({k[len(sub) + 1:]: tuple(s) for k, s in ref_layout.items()
                                                      if k.startswith(sub + ".")}))

    code = RefSynthesizerTrn.__init__.__code__
    assert list(code.co_varnames[1:code.co_argcount]) == surface["init_params"]

    def sequence_mask(length, max_length):
        return torch.arange(max_length, dtype=length.dtype, device=length.device)[None] < length[:, None]

    monkeypatch.setitem(sys.modules, "utils", types.SimpleNamespace(f0_to_coarse=f0_to_coarse))
    ref_models = types.SimpleNamespace(SynthesizerTrn=RefSynthesizerTrn, commons=types.SimpleNamespace(sequence_mask=sequence_mask))
    cls = models.patch_reference(ref_models)
    assert ref_models.SynthesizerTrn is cls and issubclass(cls, RefSynthesizerTrn)
    net = cls(1025, 20, **_model_kwargs()).eval()
    missing = net.load_state_dict(sd, strict=False)
    assert all(k.startswith(("enc_q.", "f0_decoder.")) for k in missing.missing_keys)
    c, f0, uv, sid = synth.golden_inputs(cfg, "b1_t33")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        net.infer(c, f0, uv, g=sid)
    # with the tail stubbed the patched prefix must be exactly the reference's prefix sequence (models.py:495-531) on the
    # class's own modules, and reproduce the reference fixture; the stand-in's enc_p is this package's restatement, which
    # the oracle tests hold to 1e-5 of the oracle and the oracle to 2e-5 of the reference
    gold = np.load(os.path.join(ROOT, "tests", "golden", "ref_infer_b1_t33.npz"))
    seen = {}

    def fake_tail(self, z_p, c_mask, g, f0_):
        seen["z_p"] = z_p.clone()
        return torch.zeros(z_p.shape[0], 1, z_p.shape[2] * 512)
    cls._run_tail = fake_tail
    net.infer(c, f0, uv, g=sid, noice_scale=0.4)
    with torch.no_grad():
        torch.manual_seed(52468)
        x_mask = torch.ones(1, 1, c.shape[2])
        x = net.pre(c) * x_mask + net.emb_uv(uv.long()).transpose(1, 2)
        z_want = net.enc_p(x, x_mask, f0=f0_to_coarse(f0), noice_scale=0.4)[0]
    assert torch.equal(seen["z_p"], z_want)
    assert torch.allclose(seen["z_p"], torch.from_numpy(gold["z_p"]), atol=3e-5)


def test_vocoder_surface_matches_reference_layout(tmp_path):
    """sovits_b200.nsf_hifigan mirrors vdecoder/nsf_hifigan/models.py: load_model(path) reads config.json next to the
    checkpoint, the module's state_dict has the reference's keys, and it refuses CPU tensors."""
    from sovits_b200 import nsf_hifigan
    vcfg = nsf_hifigan.cfg_from_h(synth.VOCODER_H)
    vsd = synth.synth_vocoder_state_dict(vcfg)
    with open(tmp_path / "config.json", "w") as f:
        json.dump(synth.VOCODER_H, f)
    torch.save({"generator": vsd}, tmp_path / "model")
    gen, h = nsf_hifigan.load_model(str(tmp_path / "model"), device="cpu")
    assert h.num_mels == 128 and gen.upp == 512
    own = gen.state_dict()
    assert set(own) == set(vsd) and torch.equal(own["ups.1.weight_v"], vsd["ups.1.weight_v"])
    mel, f0 = synth.synth_vocoder_inputs(vcfg, 1, 8)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        gen(mel, f0)


def test_frontend_weight_caches_follow_parameter_updates():
    """The fused q/k/v projection and the tap-stacked FFN matrices are cached per module; a load_state_dict (in-place copy,
    bumps the tensor version) or a dtype/device move must invalidate them."""
    from sovits_b200.frontend import RelEncoder
    torch.manual_seed(3)
    a, b = RelEncoder(192, 768, 2, 2, 3).eval(), RelEncoder(192, 768, 2, 2, 3).eval()
    x, m = torch.randn(2, 192, 30), torch.ones(2, 1, 30)
    with torch.no_grad():
        ya0, yb = a(x, m, True), b(x, m, True)
        assert float((ya0 - yb).abs().max()) > 1e-3            # different random weights
        a.load_state_dict(b.state_dict())
        ya1 = a(x, m, True)
        assert torch.equal(ya1, yb)                             # caches rebuilt from the new weights
        a.double()
        ya2 = a(x.double(), m.double(), True)
        assert ya2.dtype == torch.float64 and float((ya2.float() - yb).abs().max()) < 1e-4
