"""Mirror of the live part of reference model/Preprocessing.py: DynamicRNN (:7-45), InputUnitLinguisticDynamic (:89-127)
and VisualAppearanceEncoder (:191-234).

The appearance encoder (70-76 % of the model's FLOPs, SURVEY.md §8a) runs entirely in the library: one prologue pass and ONE
persistent tcgen05 launch for the W_ih product of both directions plus the 16 recurrent steps (dvgr_lstm_seq_fwd). The question
encoder's two BiLSTMs run on the same kernel (4 directions, length-masked in the cell epilogue), which removes cuDNN, the
pack/unpack round trip and the host sync on question_len from the step (SURVEY.md §8f.1). Clip features may arrive as fp32
(the reference's format) or as bf16 (stored / shipped at half the bytes)."""
import torch
import torch.nn as nn
from torch.nn import functional as F

from dualvgr_videoqa_b200 import autograd as ag


class DynamicRNN(nn.Module):
    """Length-aware RNN: packs by length, runs the cuDNN RNN, re-pads to max_num_frames; returns (outputs, final state)."""

    def __init__(self, input_size, hidden_size, num_layers=1, bias=True, batch_first=False, dropout=0,
                 bidirectional=False, rnn_encoder='GRU'):
        super().__init__()
        self.batch_first = batch_first
        self.rnn = getattr(nn, rnn_encoder)(input_size, hidden_size, num_layers=num_layers, bias=bias,
                                            batch_first=batch_first, dropout=dropout if num_layers > 1 else 0,
                                            bidirectional=bidirectional)
        self.bidirectional = bidirectional

    def forward(self, x, seq_len, max_num_frames):
        lengths = seq_len.detach().to("cpu", torch.int64)
        packed = nn.utils.rnn.pack_padded_sequence(x, lengths, batch_first=self.batch_first, enforce_sorted=False)
        out, state = self.rnn(packed)
        if isinstance(state, tuple):
            state = state[0]
        out, _ = nn.utils.rnn.pad_packed_sequence(out, batch_first=self.batch_first, total_length=max_num_frames)
        if self.bidirectional:
            state = torch.cat([state[0], state[1]], -1)
        return out, state


class InputUnitLinguisticDynamic(nn.Module):
    def __init__(self, vocab_size, wordvec_dim=300, rnn_dim=512, bidirectional=True, textual_encoder='LSTM'):
        super().__init__()
        self.bidirectional = bidirectional
        if bidirectional:
            rnn_dim = rnn_dim // 2
        self.encoder_embed = nn.Embedding(vocab_size, wordvec_dim)
        self.tanh = nn.Tanh()
        self.concatRNN = DynamicRNN(wordvec_dim, rnn_dim, num_layers=1, bias=True, batch_first=True, dropout=0.15,
                                    bidirectional=bidirectional, rnn_encoder=textual_encoder)
        self.encoder = getattr(nn, textual_encoder)(wordvec_dim, rnn_dim, batch_first=True, bidirectional=bidirectional)
        self.embedding_dropout = nn.Dropout(p=0.15)
        self.final_dropout = nn.Dropout(0.18)

    def _lstm_params(self):
        params = []
        for m in (self.concatRNN.rnn, self.encoder):
            params += [m.weight_ih_l0, m.weight_hh_l0, m.bias_ih_l0, m.bias_hh_l0,
                       m.weight_ih_l0_reverse, m.weight_hh_l0_reverse, m.bias_ih_l0_reverse, m.bias_hh_l0_reverse]
        return params

    def launch(self, questions, qlen32):
        """Launches the input unit's forward kernels (embedding + dropout + tanh, both BiLSTMs as one 4-direction recurrence)
        WITHOUT creating its autograd node; fused() adopts the result later (fused_stack.QuestionInputFn.launch explains why)."""
        from dualvgr_videoqa_b200 import fused_stack as fs
        if not (self.bidirectional and isinstance(self.encoder, nn.LSTM)):
            raise NotImplementedError("the sm_100a question encoder is the bidirectional LSTM pair DualVGR builds")
        p_emb = self.embedding_dropout.p if self.training else 0.0
        return (float(p_emb), fs.QuestionInputFn.launch(float(p_emb), questions, qlen32, self.encoder_embed.weight,
                                                        self._lstm_params()))

    def fused(self, questions, qlen32, launched=None):
        """Whole input unit as ONE autograd Function (fused_stack.QuestionInputFn). -> (question_embedding [B,D] bf16,
        words [B,L,Wp] bf16 zero-padded, per-token states [B*L, D] bf16); the first and last are column slices of wider
        buffers (valid GEMM operands). launched: the result of launch() when the kernels already went out."""
        from dualvgr_videoqa_b200 import fused_stack as fs
        cfg = launched if launched is not None else self.launch(questions, qlen32)
        dq, q, words = fs.QuestionInputFn.apply(cfg, questions, qlen32, self.encoder_embed.weight, *self._lstm_params())
        return ag.dropout(q, self.final_dropout.p, self.training), words, dq

    def forward(self, questions, question_len):
        """-> (question_embedding [B,D] bf16, words [B,L,W] fp32, per-token states [B,L,D] bf16, zero rows at padded
        positions). The embedding lookup / dropout / tanh are three tiny PyTorch ops; both BiLSTMs run as one fused
        4-direction recurrence in the library (no pack_padded_sequence, no host sync on question_len)."""
        words = self.tanh(self.embedding_dropout(self.encoder_embed(questions)))
        if not (self.bidirectional and isinstance(self.encoder, nn.LSTM)):
            raise NotImplementedError("the sm_100a question encoder is the bidirectional LSTM pair DualVGR builds")
        r, e = self.concatRNN.rnn, self.encoder
        params = []
        for m in (r, e):
            params += [m.weight_ih_l0, m.weight_hh_l0, m.bias_ih_l0, m.bias_hh_l0,
                       m.weight_ih_l0_reverse, m.weight_hh_l0_reverse, m.bias_ih_l0_reverse, m.bias_hh_l0_reverse]
        dq, q = ag.QuestionEncoderFn.apply(words.float(), question_len.to(torch.int32), *params)
        return ag.dropout(q, self.final_dropout.p, self.training), words, dq


class VisualAppearanceEncoder(nn.Module):
    def __init__(self, appearance_dim=2048, module_dim=512, bidirectional=True):
        super().__init__()
        if not bidirectional:
            raise NotImplementedError("the sm_100a appearance encoder is the bidirectional one DualVGR builds")
        self.input_dim, self.bidirectional, self.module_dim = appearance_dim, bidirectional, module_dim
        self.tanh = nn.Tanh()
        self.encoder = nn.LSTM(appearance_dim, module_dim // 2, batch_first=False, bidirectional=True)
        self.embedding_dropout = nn.Dropout(p=0.15)
        self.finalvisual_dropout = nn.Dropout(p=0.18)

    def forward(self, appearance_clips, out=None, rows=None, err=None):
        """[B, N, F, Dv] fp32 -> [B, N, module_dim] bf16 (final forward / backward hidden states, concatenated).
        out: optional preallocated [B*N, module_dim] bf16 buffer for the result.
        rows: optional [B] int32 video rows; appearance_clips is then a device-resident store [V, N, F, Dv] (fp32 / bf16)
        read at those rows inside the prologue (err: its sticky [1] int32 out-of-range word, loader.DeviceFeatureStore)."""
        e = self.encoder
        x = appearance_clips if appearance_clips.dtype == torch.bfloat16 else appearance_clips.float()   # bf16-stored features pass through
        return ag.AppearanceEncoderFn.apply(
            x, e.weight_ih_l0, e.weight_hh_l0, e.bias_ih_l0, e.bias_hh_l0,
            e.weight_ih_l0_reverse, e.weight_hh_l0_reverse, e.bias_ih_l0_reverse, e.bias_hh_l0_reverse,
            self.embedding_dropout.p, self.finalvisual_dropout.p, self.training, (out,) if out is not None else None,
            rows, err)
