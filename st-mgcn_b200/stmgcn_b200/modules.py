"""Host-side mirror of the reference's ``nn.Module`` surface (the drop-in boundary, SURVEY.md section 8(b)).

Same class names, constructor signatures, parameter names / shapes / creation order / init, ``forward``
signatures and ``state_dict`` keys as ``/root/reference/GCN.py`` and ``/root/reference/STMGCN.py`` -- so
``Main.py`` and ``Model_Trainer.py`` run unchanged and checkpoints interchange -- but every ``forward``
runs the sm_100a kernels of ``libstmgcn_b200.so`` (no torch einsum / nn.LSTM execution, no CPU path).
"""
from __future__ import annotations

import os
from typing import List, Optional

import torch
from torch import nn

from . import _lib, ops
from .graph import ChebSupports, supports_from_dense


_BRANCH_STREAMS = {}


def _graph_streams_enabled() -> bool:
    """One CUDA stream per graph branch in ``ST_MGCN.forward`` (``STMGCN_GRAPH_STREAMS=0`` runs them on one stream)."""
    return os.environ.get("STMGCN_GRAPH_STREAMS", "1") != "0"


def _act_code(activation_module) -> Optional[int]:
    """Kernel-side activation code, or None when the module must be applied by torch."""
    if activation_module is None:
        return _lib.ACT_NONE
    if type(activation_module) is nn.ReLU:
        return _lib.ACT_RELU
    return None


class GCN(nn.Module):
    """Drop-in for ``GCN.GCN`` (reference ``GCN.py:7-46``).  ``K`` is the NUMBER OF SUPPORTS."""

    def __init__(self, K: int, input_dim: int, hidden_dim: int, bias=True, activation=nn.ReLU):
        super().__init__()
        self.K = K
        self.input_dim = input_dim
        self.hidden_dim = hidden_dim
        self.bias = bias
        self.activation = activation() if activation is not None else None
        self.init_params(n_supports=K)

    def init_params(self, n_supports: int, b_init=0):
        # same creation order and initialisers as GCN.py:17-22 (same seed => same parameters)
        self.W = nn.Parameter(torch.empty(n_supports * self.input_dim, self.hidden_dim), requires_grad=True)
        nn.init.xavier_normal_(self.W)
        if self.bias:
            self.b = nn.Parameter(torch.empty(self.hidden_dim), requires_grad=True)
            nn.init.constant_(self.b, val=b_init)

    def forward_node_major(self, sset, x_nm: torch.Tensor) -> torch.Tensor:
        """x (N,B,p) node-major -> (N,B,hidden) node-major (internal fast path, no permutes)."""
        code = _act_code(self.activation)
        bias = self.b if self.bias else None
        out = ops.ChebGCN.apply(x_nm, self.W, bias, sset, _lib.ACT_NONE if code is None else code)
        return self.activation(out) if code is None else out

    def forward(self, A, x: torch.Tensor):
        """``A``: (K, N, N) supports (dense tensor as in the reference, or ``ChebSupports``);
        ``x``: (batch, N, input_dim) -> (batch, N, hidden_dim).  Reference ``GCN.py:24-43``."""
        assert self.K == A.shape[0]
        sset = supports_from_dense(A)
        x_nm = x.permute(1, 0, 2).contiguous()
        return self.forward_node_major(sset, x_nm).permute(1, 0, 2)

    def __repr__(self):
        return self.__class__.__name__ + f'({self.K} * input {self.input_dim} -> hidden {self.hidden_dim})'


class CG_LSTM(nn.Module):
    """Drop-in for ``STMGCN.CG_LSTM`` (reference ``STMGCN.py:7-57``)."""

    def __init__(self, seq_len: int, n_nodes: int, input_dim: int, lstm_hidden_dim: int, lstm_num_layers: int,
                 K: int, gconv_use_bias: bool, gconv_activation=nn.ReLU):
        super().__init__()
        self.seq_len = seq_len
        self.n_nodes = n_nodes
        self.input_dim = input_dim
        self.lstm_hidden_dim = lstm_hidden_dim
        self.lstm_num_layers = lstm_num_layers
        # creation order of STMGCN.py:17-22 (keeps same-seed init and state_dict keys identical)
        self.gconv_temporal_feats = GCN(K=K, input_dim=seq_len, hidden_dim=seq_len,
                                        bias=gconv_use_bias, activation=gconv_activation)
        self.fc = nn.Linear(in_features=seq_len, out_features=seq_len, bias=True)
        # nn.LSTM is kept as the PARAMETER CONTAINER only (names weight_ih_l0 ... as in the reference);
        # its forward is never called -- the recurrence runs in ops.SharedLSTM (stmgcn_lstm16_fwd/bwd, stmgcn_lstm_fwd/bwd).
        self.lstm = nn.LSTM(input_size=input_dim, hidden_size=lstm_hidden_dim,
                            num_layers=lstm_num_layers, batch_first=True)

    def _lstm_weights(self) -> List[torch.Tensor]:
        ws = []
        for l in range(self.lstm_num_layers):
            ws += [getattr(self.lstm, f"weight_ih_l{l}"), getattr(self.lstm, f"weight_hh_l{l}"),
                   getattr(self.lstm, f"bias_ih_l{l}"), getattr(self.lstm, f"bias_hh_l{l}")]
        return ws

    def forward_node_major(self, sset, xo: torch.Tensor, xt: torch.Tensor, h0=None, c0=None, want_state: bool = False):
        """xo (N,B,T,C), xt (N,B,T) node-major -> (h_top (N,B,H), h_n, c_n (L, N*B, H))."""
        gc = self.gconv_temporal_feats
        n = xt.shape[0]
        code = _act_code(gc.activation)
        if code is not None:
            pool = ops.TemporalPool.apply(xt, gc.W, gc.b if gc.bias else None, sset, code)
        else:       # exotic activation class: kernel does the GCN, torch applies the module + pooling
            pool = (xt + gc.forward_node_major(sset, xt)).sum(dim=0)
        s = ops.ContextGate.apply(pool, self.fc.weight, self.fc.bias, n)
        return ops.SharedLSTM.apply(xo, s, h0, c0, self.lstm_num_layers, self.lstm_hidden_dim, want_state,
                                    *self._lstm_weights())

    def forward(self, adj, obs_seq: torch.Tensor, hidden: tuple):
        """Reference ``STMGCN.py:24-51``: returns ``(output (B,N,H), (h_n, c_n) each (L, B*N, H))``."""
        b, t, n, c = obs_seq.shape
        sset = supports_from_dense(adj)
        xo, xt = ops.obs_to_node_major(obs_seq)
        lyr, hid = self.lstm_num_layers, self.lstm_hidden_dim
        h0 = c0 = None
        if hidden is not None:
            # reference rows are b*N + n (STMGCN.py:47); kernels use n*B + b
            h0 = hidden[0].reshape(lyr, b, n, hid).permute(0, 2, 1, 3).reshape(lyr, n * b, hid)
            c0 = hidden[1].reshape(lyr, b, n, hid).permute(0, 2, 1, 3).reshape(lyr, n * b, hid)
        h_top, h_n, c_n = self.forward_node_major(sset, xo, xt, h0, c0, want_state=True)
        to_ref = lambda v: v.reshape(lyr, n, b, hid).permute(0, 2, 1, 3).reshape(lyr, b * n, hid)
        return h_top.permute(1, 0, 2), (to_ref(h_n), to_ref(c_n))

    def init_hidden(self, batch_size: int):
        weight = next(self.parameters()).data
        hidden = (weight.new_zeros(self.lstm_num_layers, batch_size * self.n_nodes, self.lstm_hidden_dim),
                  weight.new_zeros(self.lstm_num_layers, batch_size * self.n_nodes, self.lstm_hidden_dim))
        return hidden


class ST_MGCN(nn.Module):
    """Drop-in for ``STMGCN.ST_MGCN`` (reference ``STMGCN.py:61-119``)."""

    def __init__(self, M: int, seq_len: int, n_nodes: int, input_dim: int, lstm_hidden_dim: int,
                 lstm_num_layers: int, gcn_hidden_dim: int, sta_kernel_config: dict, gconv_use_bias: bool,
                 gconv_activation=nn.ReLU):
        super().__init__()
        self.M = M
        self.sta_K = self.get_support_K(sta_kernel_config)
        self.rnn_list, self.gcn_list = nn.ModuleList(), nn.ModuleList()
        for m in range(self.M):                       # same interleaved creation order as STMGCN.py:69-77
            cglstm = CG_LSTM(seq_len=seq_len, n_nodes=n_nodes, input_dim=input_dim,
                             lstm_hidden_dim=lstm_hidden_dim, lstm_num_layers=lstm_num_layers,
                             K=self.sta_K, gconv_use_bias=gconv_use_bias, gconv_activation=gconv_activation)
            self.rnn_list.append(cglstm)
            gcn = GCN(K=self.sta_K, input_dim=lstm_hidden_dim, hidden_dim=gcn_hidden_dim,
                      bias=gconv_use_bias, activation=gconv_activation)
            self.gcn_list.append(gcn)
        self.fc = nn.Linear(in_features=gcn_hidden_dim, out_features=input_dim, bias=True)

    @staticmethod
    def get_support_K(config: dict):
        # STMGCN.py:80-91
        if config['kernel_type'] == 'localpool':
            assert config['K'] == 1
            K = 1
        elif config['kernel_type'] == 'chebyshev':
            K = config['K'] + 1
        elif config['kernel_type'] == 'random_walk_diffusion':
            K = config['K'] * 2 + 1
        else:
            raise ValueError('Invalid kernel_type. Must be one of [chebyshev, localpool, random_walk_diffusion].')
        return K

    def init_hidden_list(self, batch_size: int):
        # kept for API parity (STMGCN.py:93-98); forward() treats the zero state implicitly
        return [self.rnn_list[m].init_hidden(batch_size) for m in range(self.M)]

    def forward(self, obs_seq: torch.Tensor, sta_adj_list: list):
        """``obs_seq``: (B,T,N,C); ``sta_adj_list``: M support stacks -> (B,N,C).  ``STMGCN.py:100-119``."""
        assert len(sta_adj_list) == self.M
        xo, xt = ops.obs_to_node_major(obs_seq)          # shared by all graphs
        ssets = []
        for m in range(self.M):
            assert self.sta_K == sta_adj_list[m].shape[0]
            ssets.append(supports_from_dense(sta_adj_list[m]))
        feats = []
        if self.M > 1 and _graph_streams_enabled():
            # the M graph branches are independent until the fusion: one CUDA stream per branch keeps the device's work
            # queue full across kernel boundaries (autograd replays each branch's backward on the same stream)
            # (also under CUDA-graph capture: the fork / join below is the capturable event pattern, so the captured graph
            # keeps the three branches as parallel chains)
            main = torch.cuda.current_stream()
            start = main.record_event()
            streams = self._branch_streams(obs_seq.device)
            for m in range(self.M):
                with torch.cuda.stream(streams[m]):
                    streams[m].wait_event(start)
                    h_top, _, _ = self.rnn_list[m].forward_node_major(ssets[m], xo, xt)
                    feats.append(self.gcn_list[m].forward_node_major(ssets[m], h_top))
                xo.record_stream(streams[m])
                xt.record_stream(streams[m])
            for m in range(self.M):
                main.wait_stream(streams[m])
                feats[m].record_stream(main)
        else:
            for m in range(self.M):
                h_top, _, _ = self.rnn_list[m].forward_node_major(ssets[m], xo, xt)
                feats.append(self.gcn_list[m].forward_node_major(ssets[m], h_top))
        return ops.FuseOut.apply(self.fc.weight, self.fc.bias, *feats)

    def _branch_streams(self, device):
        # process-wide cache (not a module attribute: streams must not end up in deepcopy / pickle of the model)
        key = (device.index if device.index is not None else torch.cuda.current_device(), self.M)
        if key not in _BRANCH_STREAMS:
            _BRANCH_STREAMS[key] = [torch.cuda.Stream(device=device) for _ in range(self.M)]
        return _BRANCH_STREAMS[key]
