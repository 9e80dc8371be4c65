"""MNIST MLP driver (mirror of evaluate_mlp.py:14-95): wrap the three Linear layers, calibrate
on 5 % of the test set, evaluate, count term-pair ops and parameter bits, dump JSON.

Same flags (--wb --wt --db --dt --gs --out-file --test-batch-size).  Differences, all forced by
the environment: the MNIST test set and pretrained_models/mnist_mlp.pt are not available, so
--synthetic (default) uses seeded random 1x28x28 images and random-init weights; the
reference's broken `get_model_ops(qmodel, input_shape=...)` call (evaluate_mlp.py:88, a
TypeError as shipped) is made with a real input tensor; --no-cuda is rejected because the TR
op has no CPU path (it never did: kernels/tr_cuda.cpp:12-18)."""
import argparse
import json
from copy import deepcopy

import torch
import torch.nn as nn

from .profile_model import get_model_ops
from .tr_layer import TRLinearLayer, set_tr_tracking
from .train_mlp import MNISTMLP, test


def _swap(model, name, new):
    parent = model
    keys = name.split('.')
    for k in keys[:-1]:
        parent = parent._modules[k]
    parent._modules[keys[-1]] = new


def replace_linear_layers(model, tr_params, data_bits, data_terms, *, encoding='hese'):
    linears = [(n, m) for n, m in model.named_modules() if isinstance(m, nn.Linear)]
    for (name, layer), (weight_bits, group_size, weight_terms) in zip(linears, tr_params):
        _swap(model, name, TRLinearLayer(layer, data_bits, data_terms, weight_bits, group_size,
                                         weight_terms, encoding=encoding))
    return model


def static_linear_layer_settings(model, weight_bits, group_size, num_terms):
    return [(weight_bits, group_size, num_terms)
            for m in model.modules() if isinstance(m, nn.Linear)]


class _SyntheticMNIST(torch.utils.data.Dataset):
    def __init__(self, n, seed=0):
        g = torch.Generator().manual_seed(seed)
        self.data = torch.randn(n, 1, 28, 28, generator=g)
        self.targets = torch.randint(10, (n,), generator=g)

    def __len__(self):
        return len(self.targets)

    def __getitem__(self, i):
        return self.data[i], int(self.targets[i])


def main(argv=None):
    parser = argparse.ArgumentParser(description='TQ MNIST MLP evaluation')
    # the reference's flags (evaluate_mlp.py:43-54): one value per setting in each list
    for flag, what in (('--wb', 'weight bits'), ('--wt', 'weight terms'), ('--db', 'data bits'),
                       ('--dt', 'data terms'), ('--gs', 'group sizes')):
        parser.add_argument(flag, nargs='+', type=int, help=what)
    parser.add_argument('--test-batch-size', type=int, default=128, metavar='N')
    parser.add_argument('--no-cuda', action='store_true', default=False)
    parser.add_argument('--out-file', help='Output file')
    # additions: synthetic data (no MNIST in this image), optional weights
    parser.add_argument('--synthetic', action='store_true', default=True)
    parser.add_argument('--samples', type=int, default=2048, help='synthetic test-set size')
    parser.add_argument('--weights', default=None, help='optional state_dict (.pt)')
    parser.add_argument('--encoding', default='hese', choices=['hese', 'binary', 'booth'],
                        help='term encoding of every wrapped layer (hese = the reference)')
    args = parser.parse_args(argv)
    if args.no_cuda or not torch.cuda.is_available():
        raise SystemExit("the TR op is CUDA-only (kernels/tr_cuda.cpp:12-18): no CPU path")
    device = torch.device("cuda")
    loader = torch.utils.data.DataLoader(_SyntheticMNIST(args.samples), batch_size=args.test_batch_size,
                                         shuffle=False)
    torch.manual_seed(0)
    model = MNISTMLP()
    if args.weights:
        model.load_state_dict(torch.load(args.weights, map_location="cpu"))

    results = {'accs': [], 'tmacs': [], 'param_bits': []}
    for wb, wt, db, dt, gs in zip(args.wb, args.wt, args.db, args.dt, args.gs):
        qmodel = deepcopy(model).to(device)
        tr_params = static_linear_layer_settings(qmodel, wb, gs, wt)
        qmodel = replace_linear_layers(qmodel, tr_params, db, dt, encoding=args.encoding)
        test(args, qmodel, device, loader, pct=0.05)          # calibration pass
        set_tr_tracking(qmodel, False)
        acc = 100.0 * test(args, qmodel, device, loader)
        tmacs, param_bits = get_model_ops(qmodel, (torch.zeros(1, 1, 28, 28, device=device),))
        results['accs'].append(acc)
        results['tmacs'].append(tmacs)
        results['param_bits'].append(param_bits)
        print(wb, wt, db, dt, gs, acc, tmacs, param_bits)
    if args.out_file:
        with open(args.out_file, 'w') as fp:
            json.dump(results, fp)
    return results


if __name__ == '__main__':
    main()
