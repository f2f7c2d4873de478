"""Loss trajectory of the UNMODIFIED reference model over 20 steps of its own loop shape
(src/train.py:247-321) on a fixed synthetic batch - the expected values quoted in
tests/test_train_gpu.py::test_training_loop_follows_reference.  Build container only.

    python oracle/ref_train_loop.py
"""
import sys, os, torch, torch.nn as nn
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, 'tests'), os.path.join(ROOT, 'oracle')): sys.path.insert(0, p)
import synth
from make_golden import build_reference
torch.manual_seed(3)
mine = synth.build_model(0)
ref = build_reference(); ref.load_state_dict(mine.state_dict())
for lr, pmax in ((1e-3, 0.1), (2e-4, 0.0), (5e-5, 0.0)):
    ref.load_state_dict(mine.state_dict())
    for m in ref.modules():
        if isinstance(m, nn.Dropout): m.p = min(m.p, pmax)
    ref.train(); ref.cnn_encoder.backbone.eval()
    images, ids, mask = synth.make_inputs(8, 48, 61, [48, 30, 12, 48, 7, 25, 40, 3], H=64, W=64)
    labels = torch.tensor([0,1,2,3,4,5,6,7])
    opt = torch.optim.AdamW(ref.parameters(), lr=lr, weight_decay=0.05)
    losses=[]
    for _ in range(20):
        opt.zero_grad(); loss = nn.CrossEntropyLoss()(ref(images, ids, mask)["logits"], labels); loss.backward()
        nn.utils.clip_grad_norm_(ref.parameters(), 1.0); opt.step(); losses.append(round(loss.item(),3))
    print(lr, pmax, losses)
