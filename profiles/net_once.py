"""One forward_train + backward of the Mnih'15 Q-network (batch 256) between cudaProfilerStart /
cudaProfilerStop, after two warm-up passes -- the target of the ncu captures:

    ncu --set full --clock-control none --import-source on --profile-from-start off \
        -k regex:tc2_gemm -o net_once_report python profiles/net_once.py
"""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from agents_b200.networks import layers as L  # noqa: E402
from agents_b200.networks import q_network  # noqa: E402
from agents_b200.specs import tensor_spec  # noqa: E402

dev = torch.device('cuda:0')
obs_spec = tensor_spec.TensorSpec((84, 84, 4), torch.uint8)
act_spec = tensor_spec.BoundedTensorSpec((), torch.int32, 0, 5)
net = q_network.QNetwork(obs_spec, act_spec, preprocessing_layers=L.CastScale(255.),
                         conv_layer_params=((32, 8, 4), (64, 4, 2), (64, 3, 1)), fc_layer_params=(512,),
                         device=dev).set_seed(0)
net.create_variables()
x = torch.randint(0, 256, (256, 84, 84, 4), dtype=torch.uint8, device=dev)
dq = torch.randn(256, 6, device=dev)
for _ in range(2):
  q, tape = net.forward_train(x)
  net.backward(tape, dq)
torch.cuda.synchronize()
torch.cuda.cudart().cudaProfilerStart()
q, tape = net.forward_train(x)
net.backward(tape, dq)
torch.cuda.synchronize()
torch.cuda.cudart().cudaProfilerStop()
print('ok', float(q.abs().sum()))
