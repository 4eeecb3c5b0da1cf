"""TEST INFRASTRUCTURE: generates tests/golden/reference_checks.pt, the vectors tests/test_oracle_vs_reference.py and
tests/test_text_cond.py compare against, by running the UNMODIFIED reference (through oracle/ref_shim.py) on the CPU.
Run:  python oracle/make_golden_reference.py      (needs the reference checkout at $LFDM_REFERENCE_ROOT; fixed seeds)

Contents
  unet_tiny, unet_natops   tiny Unet3D built from a seed: digests of its parameters + inputs + outputs of
                           forward_with_cond_scale (the NATOPS variant: nearest upsample, reflect padding, learned null cond)
  init_identity            FlowDiffusion (mug128, seed 1234) with the default and the NATOPS options: parameter names in
                           order and a digest of every tensor (the weights themselves are not stored)
  model_params             the reference's config/*.yaml `model_params` (without avd_network_params)
  bert                     token ids and the reference's text.bert_embed on a tiny seeded BertModel (mean and [CLS])
"""
import hashlib
import importlib.util
import os
import sys
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle.ref_shim import REFERENCE_ROOT, import_reference  # noqa: E402
from oracle.make_golden import TINY_UNET  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden", "reference_checks.pt")
NATOPS_KW = dict(use_deconv=False, padding_mode="reflect", learn_null_cond=True)
BERT_IDS = torch.tensor([[2, 7, 9, 11, 3, 0, 0], [2, 5, 3, 0, 0, 0, 0], [2, 4, 6, 8, 10, 12, 3]])


def digest(t):
    """first 8 bytes of the sha256 of dtype, shape and raw bytes: equal digests <=> bit-identical tensors"""
    t = t.detach().cpu().contiguous()
    h = hashlib.sha256(f"{t.dtype}{tuple(t.shape)}".encode())
    h.update(t.reshape(-1).view(torch.uint8).numpy().tobytes())
    return int.from_bytes(h.digest()[:8], "little", signed=True)


def state_digests(sd):
    """parameter names in order (as one sha256) and one digest per tensor"""
    return dict(n=len(sd), keys=hashlib.sha256("\n".join(sd).encode()).hexdigest(),
                tensors=torch.tensor([digest(v) for v in sd.values()], dtype=torch.int64))


def tiny_bert():
    from transformers import BertConfig, BertModel
    torch.manual_seed(3)
    cfg = BertConfig(vocab_size=50, hidden_size=32, num_hidden_layers=2, num_attention_heads=2, intermediate_size=64,
                     max_position_embeddings=32)
    return BertModel(cfg).eval()


def unet_case(ns, seed, t, scales, **kw):
    torch.manual_seed(seed)
    unet = ns.Unet3D(**dict(TINY_UNET, **kw)).eval()
    x, cond = torch.randn(2, 11, 5, 8, 8), torch.randn(2, 24)
    out = {cs: unet.forward_with_cond_scale(x, t, cond=cond, cond_scale=cs) for cs in scales}
    return dict(seed=seed, kw=kw, params=state_digests(unet.state_dict()), x=x, t=t, cond=cond, out=out)


def main():
    import yaml
    ns = import_reference()
    torch.set_grad_enabled(False)
    torch.set_num_threads(8)        # the sum order of CPU convolutions depends on it: tests/conftest.py GOLDEN_THREADS
    g = dict(
        unet_tiny=unet_case(ns, 3, torch.tensor([999, 0]), (0.0, 1.0, 3.0)),
        unet_natops=unet_case(ns, 5, torch.tensor([500, 7]), (1.0, 2.0), **NATOPS_KW),
        init_identity=[], model_params={})
    cfg = os.path.join(REFERENCE_ROOT, "config", "mug128.yaml")
    for kw in (dict(), NATOPS_KW):
        torch.manual_seed(1234)
        r = ns.FlowDiffusion(is_train=False, sampling_timesteps=3, config_pth=cfg, pretrained_pth="", **kw)
        g["init_identity"].append(dict(kw=kw, params=state_digests(r.state_dict())))
    for name in ("mug128", "mhad128", "natops128"):
        mp = yaml.safe_load(open(os.path.join(REFERENCE_ROOT, "config", f"{name}.yaml")))["model_params"]
        mp.pop("avd_network_params", None)
        g["model_params"][name] = mp

    spec = importlib.util.spec_from_file_location("ref_text", os.path.join(REFERENCE_ROOT, "DM", "modules", "text.py"))
    R = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(R)
    R.MODEL = tiny_bert()
    g["bert"] = dict(ids=BERT_IDS, mean=R.bert_embed(BERT_IDS, return_cls_repr=False),
                     cls=R.bert_embed(BERT_IDS, return_cls_repr=True))
    R.MODEL = None
    torch.save(g, OUT)
    print(OUT, os.path.getsize(OUT))


if __name__ == "__main__":
    main()
