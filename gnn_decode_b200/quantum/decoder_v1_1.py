"""Drop-in for the model classes of the reference's quantum/decoder_v1_1.py: neural belief propagation whose learned
multiplicative weights are shared per EDGE TYPE -- `torch.matmul(m.mul(feat_onehot), W)` with a one-hot [E, nb_digits]
edge-type matrix (decoder_v1_1.py:196-205, 219-233, 261-275).  That is `m * W[type(e)]`, i.e. the neural_BP program with
per-edge weights gathered from the type tables, so it runs on the same kernels (GD_PROG_NEURAL_BP); only the parameter
shapes ([nb_digits, 1]) and state_dict keys (`layers.{2l}.W`, `layers.{2l}.W_p` -- the target_to_source layers own no
parameters --, `W`, `W_p`, `alpha`) differ.

The reference derives the edge types from the module global `H_one` (generate_PCM's second output); here they are the
keyword-only argument `edge_types` ([E] integers in [0, nb_digits), in edge order)."""
import torch

from .. import _cabi
from ..message_passing import DecoderBase, MessagePassingBase
from .neural_BP import WeightClipper  # noqa: F401  (same helper, decoder_v1_1.py:312-325)


class MessagePassing(MessagePassingBase):
    _gd_program = _cabi.PROG_NEURAL_BP

    def propagate(self, edge_index, extra=None, size=None, **kwargs):
        return self._propagate(edge_index, extra, size, kwargs)


def _types(edge_types, nb_digits):
    t = torch.as_tensor(edge_types, dtype=torch.long).reshape(-1)
    if t.numel() == 0 or int(t.min()) < 0 or int(t.max()) >= nb_digits:
        raise ValueError("edge_types must be [E] integers in [0, nb_digits=%d)" % nb_digits)
    return t


class GraphConv(MessagePassing):
    def __init__(self, flow, aggr='add', bias=True, *, edge_types, nb_digits=32):
        super(GraphConv, self).__init__(aggr, flow)
        self.flow = flow
        self.register_buffer("edge_types", _types(edge_types, nb_digits), persistent=False)
        self.n_edges = int(self.edge_types.numel())
        if self.flow == 'source_to_target':
            self.W = torch.nn.Parameter(torch.ones((nb_digits, 1)).double())
            self.W_p = torch.nn.Parameter(torch.ones((nb_digits, 1)).double())

    def forward(self, m, edge_index, x, prev=None):
        x = x if x.dim() == 2 else x.unsqueeze(-1)
        if self.flow == 'source_to_target':
            m = m.mul(self.W[self.edge_types].repeat(m.size(0) // self.n_edges, 1))
        return self.propagate(edge_index=edge_index, size=(x.size(0), x.size(0)), x=m, extra=x)

    def update(self, aggr_out):
        if self.flow == 'source_to_target':
            w = self.W_p[self.edge_types].repeat(aggr_out.size(0) // self.n_edges, 1)
            return aggr_out[:, 0].clone().unsqueeze(1) + aggr_out[:, 1].clone().unsqueeze(1).mul(w)
        return aggr_out

    _gd_builtin_update = update

    def _gd_hidden(self):
        return self.n_edges

    def _gd_update_params(self):
        if self.flow != 'source_to_target':
            return []
        with torch.no_grad():
            return [self.W_p[self.edge_types]]


class GNNI(DecoderBase):
    _gd_program = _cabi.PROG_NEURAL_BP

    def __init__(self, Nc, *, edge_types, nb_digits=32, rows=None, cols=None):
        super(GNNI, self).__init__(Nc, rows, cols)
        self.nb_digits = int(nb_digits)
        self.register_buffer("edge_types", _types(edge_types, nb_digits), persistent=False)
        self.n_edges = int(self.edge_types.numel())
        self.layers = self._make_layer()
        self.W = torch.nn.Parameter(torch.ones((nb_digits, 1)).double())
        self.W_p = torch.nn.Parameter((torch.ones((nb_digits, 1)) * 0.5).double())
        self.alpha = torch.nn.Parameter(torch.Tensor([[0]]).double())
        if rows is not None:
            self.bind_code(rows, cols)

    def _make_layer(self):
        layers = []
        for _ in range(self.Nc):
            layers.append(GraphConv("source_to_target", edge_types=self.edge_types, nb_digits=self.nb_digits))
            layers.append(GraphConv("target_to_source", edge_types=self.edge_types, nb_digits=self.nb_digits))
        return torch.nn.Sequential(*layers)

    def bind_code(self, rows, cols):
        super(GNNI, self).bind_code(rows, cols)
        for layer in self.layers:
            layer.bind_code(rows, cols)
        return self

    def _gd_hidden(self):
        return self.n_edges

    def _gd_params(self):
        """The per-edge weight vectors the NEURAL_BP kernel consumes: type tables gathered by edge type.  In training (train()
        mode, grad enabled) the gather is part of the autograd graph, so the per-edge gradients of the training backward are
        summed per type by the index's backward; in inference it runs without autograd."""
        t = self.edge_types
        with torch.set_grad_enabled(torch.is_grad_enabled() and self.training):
            out = []
            for l in range(self.Nc):
                out += [self.layers[2 * l].W[t], self.layers[2 * l].W_p[t]]
            return out + [self.W[t], self.W_p[t], self.alpha if torch.is_grad_enabled() else self.alpha.detach()]
