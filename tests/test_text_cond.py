"""CPU: text conditioning (cvpr23_lfdm_b200/dm/text.py) -- the reference's pooling arithmetic on an injected tiny BERT, the
label-table path, and the failure mode when neither weights nor table are available."""
import pytest
import torch


def test_bert_embed_matches_reference_pooling(golden):
    """same model, same padded token ids -> identical masked mean (excluding [CLS]) and [CLS] outputs as the reference
    (recorded by oracle/make_golden_reference.py)"""
    from cvpr23_lfdm_b200.dm import text as T
    from oracle.make_golden_reference import tiny_bert
    g = golden("reference_checks.pt")["bert"]
    T.MODEL = tiny_bert()
    try:
        for cls, ref in ((False, g["mean"]), (True, g["cls"])):
            got = T.bert_embed(g["ids"], return_cls_repr=cls)
            assert torch.equal(ref, got)
    finally:
        T.MODEL = None


def test_label_table_roundtrip_and_missing_label(tmp_path):
    from cvpr23_lfdm_b200.dm import text as T
    T.clear_text_embeddings()
    try:
        table = {s: torch.randn(768) for s in T.LABELS["mug"]}
        p = tmp_path / "table.pt"
        torch.save(table, p)
        T.load_text_table(str(p))
        e = T.bert_embed(T.tokenize(["fear", "anger"]))
        assert e.shape == (2, 768) and torch.equal(e[0], table["fear"]) and torch.equal(e[1], table["anger"])
        assert len(T.LABELS["mug"]) == 7 and len(T.LABELS["mhad"]) == 26 and len(T.LABELS["natops"]) == 24
        if T.TOKENIZER is None:      # no BERT vocabulary in this image: an unknown string must fail loudly, naming the ways out
            with pytest.raises(RuntimeError, match="LFDM_TEXT_TABLE"):
                T.tokenize(["not a label"])
    finally:
        T.clear_text_embeddings()
