"""Pins the oracle against the UNMODIFIED reference on inputs that are NOT in the other fixtures, and stores what the
reference computed in tests/golden/live_pin.npz, which tests/test_oracle.py compares the oracle against.

    VOICEFIXER_REFERENCE=<reference checkout> python tests/golden/live_pin.py [seed]     # prints one JSON line

Same loading recipe as make_golden.py (stub-loader + seeded synthetic checkpoints under a temporary HOME, loaded by
the reference's own VoiceFixer() / Vocoder(44100)).  Cases: analysis at T in {2, 64, 128, 257} (pad/crop edges of the
64-frame UNet grid), Vocoder.forward at odd and even T, restore_inmem mode 0 on 1.3 s, restore_inmem mode 2
(train-mode BN + the dropout masks the reference actually drew, captured by forward hooks), and the
your_vocoder_func hook (base.py:126-129).  Also the reference's own Slaney / HTK filterbank,
melscale_fbanks(1025, 0, 22050, 128, 44100, norm="slaney", mel_scale="htk") (voicefixer/tools/mel_scale.py:173-238).

The fixture keeps it small: the inputs are regenerated from the seed by inputs() (their sums are stored to prove it),
each output is stored as the fixed sample that sample() takes plus its shape, the dropout masks bit-packed and the
filterbank as its non-zeros."""
import json
import os
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
OUT = os.path.join(HERE, "live_pin.npz")
NSAMPLE = 2048
STRIDE = 1000003            # prime: k * STRIDE mod n visits NSAMPLE distinct elements spread over the whole array


def sample(a):
    a = np.asarray(a, np.float32).reshape(-1)
    if a.size <= NSAMPLE:
        return a
    return a[np.arange(NSAMPLE, dtype=np.int64) * STRIDE % a.size]


def inputs(seed):
    import torch
    from voicefixer_b200 import synthetic
    x = {}
    for T in (2, 64, 128, 257):
        x[f"analysis_T{T}"] = torch.rand(1, 1, T, 128, generator=torch.Generator().manual_seed(seed + T)) ** 4 * 30.0
    for T in (5, 12):
        x[f"vocoder_T{T}"] = torch.rand(1, 1, T, 128, generator=torch.Generator().manual_seed(seed + 500 + T)) ** 4 * 30.0
    x["wav_1.3s"] = synthetic.make_utterances(1, seconds=1.3, seed=seed + 1)[0]
    x["wav_1.6s"] = synthetic.make_utterances(1, seconds=1.6, seed=seed + 2)[0]
    return x


def oracle_outputs(x, ana, voc, masks):
    """The oracle's result for every case, keyed like the reference's in main()."""
    import torch
    from oracle import vf_oracle as O
    out = {}
    with torch.no_grad():
        for k in ("analysis_T2", "analysis_T64", "analysis_T128", "analysis_T257"):
            out[k] = O.analysis(x[k], ana)
        for k in ("vocoder_T5", "vocoder_T12"):
            out[k] = O.vocoder_forward(x[k], voc)
        wav = x["wav_1.3s"]
        out["restore_mode0_1.3s"] = O.restore_inmem(wav, ana, voc, mode=0)
        out["restore_mode2_1.6s"] = O.restore_inmem(x["wav_1.6s"], ana, voc, mode=2, drop_masks_fn=lambda T: masks)
        _, mel = O.frontend(torch.from_numpy(wav)[None], ana)
        out["hook_mel"] = O.from_log(O.analysis(mel, ana))
        out["hook_out"] = O.trim_center(O.vocoder_forward(out["hook_mel"], voc) * 0.5, wav.shape[0]).squeeze(0).numpy()
    return {k: np.asarray(v) for k, v in out.items()}


def stored_masks(g):
    import torch
    return [torch.from_numpy(np.unpackbits(g[f"mask{i}"])[: int(np.prod(g["mask_shape"]))].reshape(g["mask_shape"]).astype(bool))
            for i in (0, 1)]


def stored_filterbank(g):
    fb = np.zeros(int(np.prod(g["fb_shape"])), np.float32)
    fb[g["fb_idx"]] = g["fb_val"]
    return fb.reshape(g["fb_shape"])


def main(seed):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, HERE)
    os.environ["HOME"] = tempfile.mkdtemp(prefix="vfx_home_")
    import torch
    torch.set_num_threads(8)
    from voicefixer_b200 import synthetic
    synthetic.write_checkpoints(os.environ["HOME"], seed=0)
    ana, voc = synthetic.make_analysis_state(0), synthetic.make_vocoder_state(1)
    import ref_loader
    ref_loader.install()
    from voicefixer.base import VoiceFixer as RefVoiceFixer          # unmodified reference
    from voicefixer.vocoder.base import Vocoder as RefVocoder
    from voicefixer.tools.mel_scale import melscale_fbanks
    ref, ref_voc = RefVoiceFixer(), RefVocoder(44100)
    model = ref._model
    x = inputs(seed)

    got = {}
    with torch.no_grad():
        for k in ("analysis_T2", "analysis_T64", "analysis_T128", "analysis_T257"):
            got[k] = model(None, x[k])["mel"]
        for k in ("vocoder_T5", "vocoder_T12"):
            got[k] = ref_voc.forward(x[k], cuda=False)
        wav = x["wav_1.3s"]
        got["restore_mode0_1.3s"] = ref.restore_inmem(wav, cuda=False, mode=0)

        # mode 2 end to end: capture the masks the reference's two Dropout(0.5) drew (x2 scaling: kept <=> out != 0)
        masks, hooks = [], []
        for mod in model.generator.denoiser:
            if isinstance(mod, torch.nn.Dropout):
                hooks.append(mod.register_forward_hook(lambda _m, inp, outp: masks.append((outp != 0) | (inp[0] == 0))))
        torch.manual_seed(seed + 3)
        got["restore_mode2_1.6s"] = ref.restore_inmem(x["wav_1.6s"], cuda=False, mode=2)
        for h in hooks:
            h.remove()

        # the your_vocoder_func hook: the reference hands the callback a linear mel [1, 1, T, 128]
        seen = {}

        def my_vocoder(mel):
            seen["mel"] = mel.clone()
            return ref_voc.forward(mel, cuda=False) * 0.5
        ref2 = RefVoiceFixer()                                           # fresh module (mode 2 above moved BN running stats)
        got["hook_out"] = ref2.restore_inmem(wav, cuda=False, mode=0, your_vocoder_func=my_vocoder)
        got["hook_mel"] = seen["mel"]
    got = {k: np.asarray(v) for k, v in got.items()}
    fb = melscale_fbanks(1025, 0.0, 22050.0, 128, 44100, norm="slaney", mel_scale="htk").numpy()

    mine = oracle_outputs(x, ana, voc, masks)
    rep = {}
    for k, v in got.items():
        assert mine[k].shape == v.shape, (k, mine[k].shape, v.shape)
        a, b = mine[k].astype(np.float64), v.astype(np.float64)
        rep[k] = float(np.sqrt(np.mean((a - b) ** 2)) / (np.sqrt(np.mean(b ** 2)) + 1e-30))
    assert masks[0].shape == masks[1].shape
    fixture = dict(seed=seed, mask_shape=np.array(masks[0].shape), fb_shape=np.array(fb.shape))
    fixture.update({f"mask{i}": np.packbits(m.numpy()) for i, m in enumerate(masks)})
    fixture["fb_idx"] = np.flatnonzero(fb).astype(np.int32)
    fixture["fb_val"] = fb.reshape(-1)[fixture["fb_idx"]]
    fixture.update({"insum_" + k: np.sum(np.asarray(v, np.float64)) for k, v in x.items()})
    fixture.update({"ref_" + k: sample(v) for k, v in got.items()})
    fixture.update({"shape_" + k: np.array(v.shape) for k, v in got.items()})
    np.savez_compressed(OUT, **fixture)
    print(json.dumps(rep))


if __name__ == "__main__":
    main(int(sys.argv[1]) if len(sys.argv) > 1 else 9100)
