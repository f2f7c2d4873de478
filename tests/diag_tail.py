"""Accuracy of the fused tail (one launch) against the per-layer launches, both against the oracle (imports oracle/, so it lives under tests/)."""
import os, sys, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import mrd_b200, synth
from oracle import forward_oracle as oracle
GOLD = os.path.join(ROOT, "tests", "golden")
model = synth.build_model(0)
plain = {k: v.clone() for k, v in model.state_dict().items()}
sens = synth.sensitise(plain, 1)
model = model.to("cuda:0")


def per_layer(eng, img, txt):
    """fusion, then head + softmax: the per-layer launches (mrd_fusion_fwd, mrd_head_fwd)"""
    f = eng.fusion(img, txt, 512, 8)[0]
    l, p = eng.head(f, 10)
    return l, p, f


for wname, sd0 in (("plain", plain), ("sens", sens)):
    model.load_state_dict(sd0, strict=True)
    sd = {k: v.float() for k, v in sd0.items() if v.is_floating_point()}
    eng = model._engine()
    g = torch.Generator().manual_seed(5)
    img = torch.randn(2048, 512, generator=g); txt = torch.randn(2048, 768, generator=g) * 0.5
    with torch.no_grad():
        rf, _ = oracle.attention_fusion(sd, img, txt); rl = oracle.classification_head(sd, rf)
    rp = torch.softmax(rl, -1)
    for path in ("fused", "per-layer"):
        l, p, f = eng.fusion_head(img, txt, 512, 10, want_fused=True) if path == "fused" else per_layer(eng, img, txt)
        l, p, f = l.cpu(), p.cpu(), f.cpu()
        relf = ((f - rf).norm(dim=-1) / rf.norm(dim=-1)).max().item()
        rell = ((l - rl).norm(dim=-1) / rl.norm(dim=-1)).max().item()
        print(wname, path, "fused rel", round(relf, 5), "logit maxabs", round((l - rl).abs().max().item(), 5), "scale", round(rl.abs().max().item(), 2),
              "logit rel-L2 max", round(rell, 5), "probs maxabs", round((p - rp).abs().max().item(), 5), "probs mean", round((p - rp).abs().mean().item(), 7),
              "top1", (l.argmax(-1) == rl.argmax(-1)).float().mean().item())
for name in ["cfg1_plain_b4_s128", "cfg1_sens_b4_s128", "padded_sens_b5_s128", "padded_sens_b3_s48"]:
    fix = torch.load(os.path.join(GOLD, name + ".pt"))
    model.load_state_dict(plain if fix["weights"] == "plain" else sens, strict=True)
    images, ids, mask = synth.make_inputs(fix["B"], fix["S"], fix["seed"], fix["lengths"])
    with torch.no_grad():
        out = model(images.cuda(), ids.cuda(), mask.cuda() if mask is not None else None, return_embeddings=True)
    pl, pp, _ = per_layer(model._engine(), out["image_embedding"], out["text_embedding"])
    for path, l, p in (("fused", out["logits"], out["probs"]), ("per-layer", pl, pp)):
        print(name, path, "logits err", (l.cpu() - fix["logits"]).abs().max().item(), "probs err", (p.cpu() - fix["probs"]).abs().max().item())
