"""Wikitext-2 LSTM driver (mirror of evaluate_lstm.py:17-176): wrap nn.LSTM and the decoder
Linear, calibrate on one pass, evaluate perplexity, count term-pair ops.

Same flags (--wb --wt --db --dt --gs --out-file, model hyper-parameters).  The corpus
(train.txt is missing, .MISSING_LARGE_BLOBS) and pretrained_models/lstm.pt are unavailable, so
tokens are synthetic (uniform over the 33,278-word vocabulary) and weights random-init.
`--tied/--cuda` keep the reference's inverted store_false behaviour (evaluate_lstm.py:77-82)."""
import argparse
import json
import math
from copy import deepcopy

import torch
import torch.nn as nn

from . import profile_model
from .lstm_models.model import RNNModel
from .tr_layer import TRLinearLayer, TRLSTMLayer, set_tr_tracking

NTOKENS = 33278


def replace_lstm_layers(model, tr_params, data_bits, data_terms, *, encoding='hese'):
    targets = [(n, m) for n, m in model.named_modules() if isinstance(m, (nn.Linear, nn.LSTM))]
    for (name, layer), (weight_bits, group_size, weight_terms) in zip(targets, tr_params):
        cls = TRLSTMLayer if isinstance(layer, nn.LSTM) else TRLinearLayer
        parent = model
        keys = name.split('.')
        for k in keys[:-1]:
            parent = parent._modules[k]
        parent._modules[keys[-1]] = cls(layer, data_bits, data_terms, weight_bits, group_size,
                                        weight_terms, encoding=encoding)
    return model


def static_lstm_layer_settings(model, weight_bits, group_size, num_terms):
    return [(weight_bits, group_size, num_terms)
            for m in model.modules() if isinstance(m, (nn.Linear, nn.LSTM))]


def convert_model(model, tr_params, data_bits, data_terms, *, encoding='hese'):
    return replace_lstm_layers(deepcopy(model), tr_params, data_bits, data_terms, encoding=encoding)


def repackage_hidden(h):
    return h.detach() if isinstance(h, torch.Tensor) else tuple(repackage_hidden(v) for v in h)


def main(argv=None):
    parser = argparse.ArgumentParser(description='TQ LSTM language-model evaluation')
    parser.add_argument('--model', type=str, default='LSTM')
    parser.add_argument('--emsize', type=int, default=650)
    parser.add_argument('--nhid', type=int, default=650)
    parser.add_argument('--nlayers', type=int, default=2)
    parser.add_argument('--bptt', type=int, default=35)
    parser.add_argument('--dropout', type=float, default=0.5)
    parser.add_argument('--tied', action='store_false')
    parser.add_argument('--seed', type=int, default=1111)
    parser.add_argument('--cuda', action='store_false')
    for flag, what in (('--wb', 'weight bits'), ('--wt', 'weight terms'), ('--db', 'data bits'),
                       ('--dt', 'data terms'), ('--gs', 'group sizes')):       # one value per setting
        parser.add_argument(flag, nargs='+', type=int, help=what)
    parser.add_argument('--out-file', help='Output file')
    parser.add_argument('--eval-batch-size', type=int, default=10)
    parser.add_argument('--encoding', default='hese', choices=['hese', 'binary', 'booth'],
                        help='term encoding of every wrapped layer (hese = the reference)')
    parser.add_argument('--tokens', type=int, default=35 * 10 * 4 + 10, help='synthetic test tokens')
    args = parser.parse_args(argv)
    if not args.cuda or not torch.cuda.is_available():
        raise SystemExit("the TR op is CUDA-only: no CPU path")
    device = torch.device("cuda")
    torch.manual_seed(args.seed)
    bsz = args.eval_batch_size
    stream = torch.randint(NTOKENS, (args.tokens,))
    nbatch = stream.size(0) // bsz
    test_data = stream[: nbatch * bsz].view(bsz, -1).t().contiguous().to(device)
    model = RNNModel(args.model, NTOKENS, args.emsize, args.nhid, args.nlayers, args.dropout,
                     args.tied).to(device)
    criterion = nn.NLLLoss()

    def get_batch(source, i):
        seq_len = min(args.bptt, len(source) - 1 - i)
        return source[i:i + seq_len], source[i + 1:i + 1 + seq_len].view(-1)

    def evaluate(m, source):
        m.eval()
        total = 0.
        hidden = m.init_hidden(bsz)
        with torch.no_grad():
            for i in range(0, source.size(0) - 1, args.bptt):
                data, targets = get_batch(source, i)
                output, hidden = m(data, hidden)
                hidden = repackage_hidden(hidden)
                total += len(data) * criterion(output, targets).item()
        return total / (len(source) - 1)

    results = {'ppls': [], 'tmacs': [], 'param_bits': []}
    for wb, wt, db, dt, gs in zip(args.wb, args.wt, args.db, args.dt, args.gs):
        tr_params = static_lstm_layer_settings(model, wb, gs, wt)
        qmodel = convert_model(model, tr_params, db, dt, encoding=args.encoding)
        evaluate(qmodel, test_data)                      # calibration pass
        set_tr_tracking(qmodel, False)
        loss = evaluate(qmodel, test_data)
        inputs = (get_batch(test_data, 0)[0], model.init_hidden(bsz))
        tmacs, param_bits = profile_model.get_model_ops(qmodel, inputs=inputs)
        ppl = math.exp(loss)
        results['ppls'].append(ppl)
        results['tmacs'].append(tmacs)
        results['param_bits'].append(param_bits)
        print(wb, wt, db, dt, gs, ppl, tmacs, param_bits)
    if args.out_file:
        with open(args.out_file, 'w') as fp:
            json.dump(results, fp)
    return results


if __name__ == '__main__':
    main()
