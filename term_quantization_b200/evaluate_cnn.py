"""ImageNet-CNN driver (mirror of evaluate_cnn.py:13-130): wrap every conv but the first,
calibrate the activation scale factors on 5 % of the data, validate, count term-pair ops;
sweeps plain quantisation (6-9 bit) and TR (g=8, alpha in {12,16,20,24}, data_terms in {2,3,4}).

Same positional/flag CLI.  There is no ImageNet and no pretrained checkpoint here, so the
loader is synthetic (util.synthetic_loader) and weights are random-init; `--quick` runs a
single TR setting.  `nn.DataParallel` (evaluate_cnn.py:33) is replaced by running on the
selected GPU; the multi-GPU path is inference.ShardedInference (one process per GPU)."""
import argparse
import json

import torch
import torch.nn as nn

from . import cnn_models, profile_model, tr_layer, util


def compute_avg_terms(tr_params):
    alphas = [terms / group for _, group, terms in tr_params[1:]]
    return sum(alphas) / len(alphas)


def eval_model(args, model, val_loader, criterion, weight_bits, group_size, weight_terms, data_bits,
               data_terms):
    tr_params = cnn_models.static_conv_layer_settings(model, weight_bits, group_size, weight_terms)
    avg_terms = compute_avg_terms(tr_params)
    qmodel = cnn_models.convert_model(model, tr_params, data_bits, data_terms,
                                      encoding=getattr(args, "encoding", "hese"))
    x = torch.zeros(1, 3, 224, 224, device=next(qmodel.parameters()).device)
    tmacs, params = profile_model.get_model_ops(qmodel, (x,))
    # profile ran one tracking-mode forward on zeros; restart the histograms before calibrating
    for m in qmodel.modules():
        if isinstance(m, tr_layer.LinearQuantize):
            m.hist_bins.zero_()
    util.validate(val_loader, qmodel, criterion, args, verbose=args.verbose, pct=0.05)
    tr_layer.set_tr_tracking(qmodel, False)
    _, acc = util.validate(val_loader, select_engine(qmodel, getattr(args, "engine", "float")), criterion, args,
                           verbose=args.verbose)
    return acc, tmacs, avg_terms, params


def select_engine(qmodel, engine):
    """How the calibrated model runs the validation pass.
    'float'   -- the reference's path: TR kernels + cuDNN fp32 conv on dequantised tensors (tr_layer.py:124-126);
    'tcgen05' -- every supported wrapped conv on integer term codes with the tcgen05 kernel, module tree unchanged;
    'fused'   -- the fused executor of the architecture (fused.FusedResNet for ResNets (BasicBlock or Bottleneck), fused.FusedVGG,
                 fused.FusedMobileNet): BN / residual / ReLU(6) / next encode in the conv epilogue, depthwise convs code
                 to code;
    'auto'    -- 'fused' where the topology allows it, else 'tcgen05'.
    On the tensor-core engines every conv's accumulator is exact by contract (conv_codes.plan_weight)."""
    if engine == "float":
        return qmodel
    from . import fused
    qmodel = qmodel.to(memory_format=torch.channels_last)
    if engine in ("fused", "auto"):
        errors = []
        for cls in (fused.FusedResNet, fused.FusedVGG, fused.FusedMobileNet):
            try:
                return cls(qmodel)
            except (NotImplementedError, AttributeError, IndexError, TypeError) as e:
                errors.append(f"{cls.__name__}: {e}")
        if engine == "fused":
            raise NotImplementedError("no fused executor for this architecture: " + "; ".join(errors))
    tr_layer.use_tensor_cores(qmodel)
    return qmodel


def main(argv=None):
    parser = argparse.ArgumentParser(description='TQ CNN evaluation')
    parser.add_argument('val_dir', nargs='?', default=None,
                        help='dataset root holding imagenet/val (evaluate_cnn.py:50); synthetic images when absent')
    parser.add_argument('-a', '--arch', default='resnet18', choices=cnn_models.model_names() + cnn_models.resnet_names())
    parser.add_argument('-j', '--workers', default=0, type=int)
    parser.add_argument('-b', '--batch-size', default=256, type=int)
    parser.add_argument('-p', '--print-freq', default=10, type=int)
    parser.add_argument('--gpu', default=0, type=int)
    parser.add_argument('-v', '--verbose', action='store_true')
    parser.add_argument('--images', default=1024, type=int, help='synthetic validation images')
    parser.add_argument('--quick', action='store_true', help='one TR setting only')
    parser.add_argument('--engine', default='float', choices=['float', 'tcgen05', 'fused', 'auto'],
                        help='how the calibrated model runs (float = the reference path)')
    parser.add_argument('--encoding', default='hese', choices=['hese', 'binary', 'booth'],
                        help='term encoding of every wrapped layer (hese = the reference)')
    parser.add_argument('--out-file', default=None)
    args = parser.parse_args(argv)
    if not torch.cuda.is_available():
        raise SystemExit("the TR op is CUDA-only: no CPU path")
    torch.cuda.set_device(args.gpu)
    val_loader = util.get_imagenet_validation(args)        # evaluate_cnn.py:62; synthetic without the dataset
    criterion = nn.CrossEntropyLoss().cuda(args.gpu)
    torch.manual_seed(0)
    if args.arch == 'efficientnet_b0':
        model = cnn_models.efficientnet_b0(pretrained=False)
    else:
        model = getattr(cnn_models, args.arch)(weights=None)
    model = model.cuda(args.gpu).eval()

    keys = ['quant', 'tr-data2', 'tr-data3', 'tr-data4']
    results = {k: {'accs': [], 'tmacs': [], 'avg_terms': [], 'params': []} for k in keys}

    def record(key, res):
        acc, tmacs, avg_terms, params = res
        print(key, tmacs, acc)
        for name, v in zip(('accs', 'tmacs', 'avg_terms', 'params'), (acc, tmacs, avg_terms, params)):
            results[key][name].append(v)

    if not args.quick:
        for weight_bits in (6, 7, 8, 9):                      # plain quantisation
            record('quant', eval_model(args, model, val_loader, criterion, weight_bits, 1, 9, 9, 9))
    for data_terms in ((3,) if args.quick else (2, 3, 4)):    # term revealing
        for weight_terms in ((12,) if args.quick else (12, 16, 20, 24)):
            record('tr-data{}'.format(data_terms),
                   eval_model(args, model, val_loader, criterion, 9, 8, weight_terms, 9, data_terms))
    out = args.out_file or 'results/{}-results.json'.format(args.arch)
    try:
        with open(out, 'w') as fp:
            json.dump(results, fp)
    except OSError:
        pass
    return results


if __name__ == '__main__':
    main()
