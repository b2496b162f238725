"""Helper script of the drop-in tests: the training loop of the reference's scripts/torch/train.py:95-233 restated on
`import voxelmorph as vxm` (argument handling cut down to what the tests pass), run by the `-m gpu` tests of
tests/test_shim.py."""
import argparse
import json
import os

import numpy as np
import torch

os.environ['NEURITE_BACKEND'] = 'pytorch'
os.environ['VXM_BACKEND'] = 'pytorch'
import voxelmorph as vxm  # noqa: E402

parser = argparse.ArgumentParser()
parser.add_argument('--img-list', required=True)
parser.add_argument('--model-dir', default='models')
parser.add_argument('--gpu', default='0')
parser.add_argument('--batch-size', type=int, default=1)
parser.add_argument('--epochs', type=int, default=1)
parser.add_argument('--steps-per-epoch', type=int, default=3)
parser.add_argument('--lr', type=float, default=1e-4)
parser.add_argument('--enc', type=int, nargs='+')
parser.add_argument('--dec', type=int, nargs='+')
parser.add_argument('--int-steps', type=int, default=7)
parser.add_argument('--int-downsize', type=int, default=2)
parser.add_argument('--image-loss', default='mse')
parser.add_argument('--lambda', type=float, dest='weight', default=0.01)
parser.add_argument('--report', help='json file: per-step losses, parameter checksum (test instrumentation)')
args = parser.parse_args()

train_files = vxm.py.utils.read_file_list(args.img_list)
generator = vxm.generators.scan_to_scan(train_files, batch_size=args.batch_size, bidir=False, add_feat_axis=True)
inshape = next(generator)[0][0].shape[1:-1]
os.makedirs(args.model_dir, exist_ok=True)
device = 'cuda'
os.environ['CUDA_VISIBLE_DEVICES'] = args.gpu
enc_nf = args.enc if args.enc else [16, 32, 32, 32]
dec_nf = args.dec if args.dec else [32, 32, 32, 32, 32, 16, 16]
model = vxm.networks.VxmDense(inshape=inshape, nb_unet_features=[enc_nf, dec_nf], bidir=False, int_steps=args.int_steps,
                              int_downsize=args.int_downsize)
model.to(device)
model.train()
optimizer = torch.optim.Adam(model.parameters(), lr=args.lr)
image_loss_func = vxm.losses.NCC().loss if args.image_loss == 'ncc' else vxm.losses.MSE().loss
losses = [image_loss_func, vxm.losses.Grad('l2', loss_mult=args.int_downsize).loss]
weights = [1, args.weight]
history = []
for epoch in range(args.epochs):
    model.save(os.path.join(args.model_dir, '%04d.pt' % epoch))
    for step in range(args.steps_per_epoch):
        inputs, y_true = next(generator)
        inputs = [torch.from_numpy(d).to(device).float().permute(0, 4, 1, 2, 3) for d in inputs]
        y_true = [torch.from_numpy(d).to(device).float().permute(0, 4, 1, 2, 3) for d in y_true]
        y_pred = model(*inputs)
        loss = 0
        for n, loss_function in enumerate(losses):
            loss = loss + loss_function(y_true[n], y_pred[n]) * weights[n]
        history.append(loss.item())
        optimizer.zero_grad()
        loss.backward()
        optimizer.step()
model.save(os.path.join(args.model_dir, '%04d.pt' % args.epochs))
if args.report:
    flat = torch.cat([p.detach().reshape(-1).double().cpu() for p in model.parameters()])
    rank = int(os.environ.get('RANK', '0'))
    dp = getattr(model, '_dp', None)
    with open(args.report + '.%d' % rank, 'w') as f:
        json.dump(dict(losses=history, param_sum=float(flat.sum()), param_abs=float(flat.abs().sum()), rank=rank,
                       allreduces=None if dp is None else dp.allreduces, engine=vxm.networks.ops.resolve_engine(model)), f)
print('done', history, flush=True)
