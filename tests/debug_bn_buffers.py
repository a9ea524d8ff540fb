import os
import sys
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path[:0] = [os.path.dirname(HERE), os.path.join(os.path.dirname(HERE), 'lfd-a-light-and-fast-detector_b200'), HERE]
import torch
from helpers import synth_model
import synth
from aten_train_reference import train_forward as aten_train_forward
for cfg in ('TL_L','WIDERFACE_L'):
    model,_=synth_model(cfg, cls_bias=-2.0); ref,_=synth_model(cfg, cls_bias=-2.0); emu,_=synth_model(cfg, cls_bias=-2.0)
    model.cuda().train(); ref.cuda().train(); emu.cuda().train()
    x = synth.synth_input(2, 184, 248).cuda()
    with torch.no_grad():
        model(x); aten_train_forward(ref, x); aten_train_forward(emu, x, emulate_bf16=True)
    rows=[]
    for (name, a), (_, b), (_, e) in zip(model.named_buffers(), ref.named_buffers(), emu.named_buffers()):
        if a.dtype.is_floating_point:
            d=float((a-b).abs().max()/b.abs().max().clamp(min=1e-6)); de=float((e-b).abs().max()/b.abs().max().clamp(min=1e-6)); dn=float((a-e).abs().max()/b.abs().max().clamp(min=1e-6))
            rows.append((d,de,dn,name,float(b.abs().max())))
    rows.sort(reverse=True)
    for r in rows[:6]: print(cfg, 'native-fp32 %.2e emu-fp32 %.2e native-emu %.2e %s max|b| %.3g'%r)
