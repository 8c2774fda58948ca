"""Host side of the packed variable-length path: the tile planner of the varlen attention kernels
(xfm_attention_varlen_plan) and the parameter layout / checkpoint import of text_classification.RobertaForSequenceClassification.
No GPU needed."""
import numpy as np
import pytest
import torch


@pytest.fixture(scope="module")
def L():
    from xfm_b200 import lib

    lib.load()
    return lib


def check_plan(lengths, cu, tiles):
    ln = np.asarray(lengths)
    assert cu.tolist() == [0] + np.cumsum(ln).tolist()
    t = tiles.tolist()
    assert t[0] == 0 and t[-1] == len(ln) and all(a < b for a, b in zip(t, t[1:]))   # in order, every sequence once
    for a, b in zip(t, t[1:]):
        rows = int(ln[a:b].sum())
        assert rows <= 128
        if b < len(ln):
            assert rows + int(ln[b]) > 128, "the tile could take the next sequence"


@pytest.mark.parametrize("seed", range(20))
def test_plan_random(L, seed):
    rng = np.random.default_rng(seed)
    n = int(rng.integers(1, 400))
    hi = int(rng.choice([2, 9, 40, 64, 129]))
    lengths = rng.integers(1, hi, n)
    cu, tiles = L.varlen_plan(lengths)
    check_plan(lengths, cu, tiles)


@pytest.mark.parametrize("lengths, n_tiles", [([1] * 300, 3), ([1] * 128, 1), ([128] * 5, 5), ([40] * 9, 3),
                                               ([40] * 10, 4), ([64, 65, 64], 3), ([127, 1, 1], 2), ([7], 1)])
def test_plan_edges(L, lengths, n_tiles):
    cu, tiles = L.varlen_plan(lengths)
    check_plan(lengths, cu, tiles)
    assert tiles.numel() - 1 == n_tiles


@pytest.mark.parametrize("lengths", [[0], [5, 0, 5], [129], [3, 200], []])
def test_plan_rejects(L, lengths):
    with pytest.raises(RuntimeError, match="code -2"):
        L.varlen_plan(lengths)


def _hf():
    return pytest.importorskip("transformers")


TINY = dict(vocab_size=120, hidden_size=128, num_hidden_layers=2, num_attention_heads=2, intermediate_size=256,
            max_position_embeddings=140, num_labels=3)
BASE = dict(vocab_size=50265, hidden_size=768, num_hidden_layers=12, num_attention_heads=12, intermediate_size=3072,
            max_position_embeddings=514, num_labels=2)


@pytest.mark.parametrize("dims", [TINY, BASE], ids=["tiny", "roberta-base"])
def test_state_dict_matches_transformers(dims):
    tr = _hf()
    from xfm_b200.text_classification import RobertaForSequenceClassification as M

    cfg = tr.RobertaConfig(**dims)
    with torch.device("meta"):
        want = {k: tuple(v.shape) for k, v in tr.RobertaForSequenceClassification(cfg).state_dict().items()}
    got = {k: tuple(v.shape) for k, v in M(cfg).state_dict().items()}
    assert got == want
    assert sorted(n for n, _ in M(cfg.to_dict()).named_parameters()) == sorted(want)


def test_from_xfm_checkpoint_maps_both_spellings(tmp_path):
    tr = _hf()
    from xfm_b200.text_classification import RobertaForSequenceClassification as M

    cfg = tr.RobertaConfig(**TINY)
    src = tr.RobertaForSequenceClassification(cfg).state_dict()
    enc = {k[len("roberta."):]: v for k, v in src.items() if k.startswith("roberta.")}
    half = sorted(enc)[::2]
    ck = {("text_encoder.roberta." + k if k in half else "text_encoder." + k): v for k, v in enc.items()}
    ck["vision_encoder.cls_token"] = torch.zeros(1, 1, 8)          # other branches of the checkpoint are ignored
    ck["text_encoder.lm_head.bias"] = torch.zeros(cfg.vocab_size)
    torch.save({"model": ck}, tmp_path / "xfm.pth")
    m = M.from_xfm_checkpoint(str(tmp_path / "xfm.pth"), cfg)
    sd = m.state_dict()
    for k, v in enc.items():
        assert torch.equal(sd["roberta." + k], v), k
    assert float(sd["classifier.dense.bias"].abs().max()) == 0.0
    assert 0.005 < float(sd["classifier.dense.weight"].std()) < 0.05   # normal(0, initializer_range = 0.02)


def test_from_pretrained_reads_config_and_weights(tmp_path):
    tr = _hf()
    from xfm_b200.text_classification import RobertaForSequenceClassification as M

    cfg = tr.RobertaConfig(**TINY)
    mlm = tr.RobertaForMaskedLM(cfg)
    cfg.to_json_file(str(tmp_path / "config.json"))
    torch.save(mlm.state_dict(), tmp_path / "pytorch_model.bin")
    m = M.from_pretrained(str(tmp_path), num_labels=1)
    assert m.num_labels == 1 and m.state_dict()["classifier.out_proj.weight"].shape == (1, cfg.hidden_size)
    sd = m.state_dict()
    for k, v in mlm.state_dict().items():
        if k.startswith("roberta.") and k in sd:
            assert torch.equal(sd[k], v), k


def test_rejects_non_64_head_dim():
    from xfm_b200.text_classification import RobertaForSequenceClassification as M

    with pytest.raises(ValueError):
        M(dict(TINY, num_attention_heads=4))
