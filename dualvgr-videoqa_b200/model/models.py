"""Mirror of reference model/models.py: DualVGR (:35-83) and DualVGRUnit_multiple (:86-173).

Same constructor arguments, forward signature, returned 7-tuple and state_dict keys/shapes as the reference, so
train.py / validate.py drive it unchanged. Differences that are fixes of environment bugs, not of arithmetic:
  * the adjacency lives on the module's own device (the reference pins it to the literal 'cuda:1', models.py:118-119);
    it is a non-persistent buffer, so it is NOT in the state_dict (as in the reference, where it is a plain attribute);
  * the per-layer GAT outputs are returned as CUDA tensors (the reference moves them to the CPU at :153-160 and
    train.py:152-153 moves them straight back with .cuda(), which is a no-op here).
"""
import numpy as np
import torch
import torch.nn as nn

from dualvgr_videoqa_b200 import autograd as ag
from dualvgr_videoqa_b200 import fused_stack as fs

from .AnswerDecoder import ContextSelfAttn, SimpleOutputUnitOpenEnded
from .Attention import AttentionSFGCN
from .GraphNN import fused_gat_layer, punishGAT
from .Preprocessing import InputUnitLinguisticDynamic, VisualAppearanceEncoder
from .fusions.fusions import MFB
from .utils import QueryAttn, QueryPunish, init_modules, pad_last

BF16 = torch.bfloat16


def normalize(mx):
    """Row-normalise a dense non-negative matrix (reference :26-33, there on a scipy sparse matrix)."""
    rowsum = mx.sum(1)
    r_inv = np.where(rowsum > 0, 1.0 / np.maximum(rowsum, 1e-300), 0.0)
    return mx * r_inv[:, None]


def build_adjacency(num_of_nodes):
    """Fully connected clip graph of reference :114-116: ones -> symmetrise -> + I -> row-normalise (dense)."""
    adj = np.ones((num_of_nodes, num_of_nodes), dtype=np.float64)
    adj = np.maximum(adj, adj.T)
    return torch.from_numpy(normalize(adj + np.eye(num_of_nodes)).astype(np.float32))


class DualVGR(nn.Module):
    def __init__(self, vision_dim=2048, module_dim=768, word_dim=300, vocab=None, num_of_nodes=8, graph_module='GCN',
                 graph_layers=1, unit_layers=2):
        super().__init__()
        self.feature_aggregation = ContextSelfAttn(module_dim)
        encoder_vocab_size = len(vocab['question_token_to_idx'])
        self.num_classes = len(vocab['answer_token_to_idx'])
        self.linguistic_input_unit = InputUnitLinguisticDynamic(vocab_size=encoder_vocab_size, wordvec_dim=word_dim,
                                                                rnn_dim=module_dim, textual_encoder='LSTM')
        self.visual_appearance_input_unit = VisualAppearanceEncoder(appearance_dim=vision_dim, module_dim=module_dim,
                                                                    bidirectional=True)
        self.visual_motion_input_unit = nn.Linear(vision_dim, module_dim)
        self.visual_input_unit = DualVGRUnit_multiple(word_dim=word_dim, module_dim=module_dim,
                                                      num_of_nodes=num_of_nodes, appearance_graph_layers=graph_layers,
                                                      motion_graph_layers=graph_layers, graph_module=graph_module,
                                                      unit_layers=unit_layers)
        self.output_unit = SimpleOutputUnitOpenEnded(module_dim=module_dim, num_answers=self.num_classes)
        init_modules(self.modules(), w_init="xavier_uniform")
        nn.init.uniform_(self.linguistic_input_unit.encoder_embed.weight, -1.0, 1.0)

    def set_precision(self, precision):
        """"bf16" (default): bf16 activations / bf16 tensor-core products with fp32 accumulation, the fast path.
        "fp32": fp32 activations, every product a 3 x bf16 split product (fp32_path.py) — the mode that meets the reference's
        fp32 results to 1e-4. The setting is process-wide (autograd.ACT): one precision per process."""
        if precision not in ("bf16", "fp32"):
            raise ValueError(f"precision must be 'bf16' or 'fp32', got {precision!r}")
        self.precision = precision
        ag.ACT[0] = torch.float32 if precision == "fp32" else BF16
        return self

    def _forward_fp32(self, video_appearance_feat, video_motion_feat, question, question_len, rows=None, err=None):
        """fp32 mode: module-by-module, fp32 activations (fp32_path.py). Same returns as forward(). With rows, the two
        feature arguments are device-resident stores read at those rows (forward_from_store)."""
        from dualvgr_videoqa_b200 import fp32_path as f32
        ag.begin_forward()
        training = self.training
        _, N, T, Dv = video_appearance_feat.shape
        B = video_appearance_feat.shape[0] if rows is None else rows.numel()
        D = self.visual_motion_input_unit.out_features
        qlen = question_len.to(torch.int32)
        lin = self.linguistic_input_unit
        words, x_tm = f32.Embed32Fn.apply(question, lin.encoder_embed.weight,
                                          float(lin.embedding_dropout.p) if training else 0.0)
        seq, last = f32.Lstm32Fn.apply(x_tm, qlen, True, *lin._lstm_params())
        dynamic_q = seq[:, :, :D]
        question_embedding = ag.dropout(last[:, D:], lin.final_dropout.p, training)
        enc = self.visual_appearance_input_unit
        seed, sid = ag._site()
        p_x = enc.embedding_dropout.p if training else 0.0
        if rows is None:
            feats = video_appearance_feat if video_appearance_feat.dtype == BF16 else video_appearance_feat.float()
            xa = ag.ops.prep_features(feats.contiguous().view(B * N * T, Dv), T, True, True, p_x, seed, sid,
                                      out_dtype=torch.float32)
        else:
            xa = ag.ops.prep_features_gather(video_appearance_feat, rows, T, True, True, p_x, seed, sid, err,
                                             out_dtype=torch.float32)
        e = enc.encoder
        _, h = f32.Lstm32Fn.apply(xa.view(T, B * N, Dv), None, False, e.weight_ih_l0, e.weight_hh_l0, e.bias_ih_l0, e.bias_hh_l0,
                                  e.weight_ih_l0_reverse, e.weight_hh_l0_reverse, e.bias_ih_l0_reverse, e.bias_hh_l0_reverse)
        app = ag.dropout(h, enc.finalvisual_dropout.p, training).view(B, N, D)
        if rows is None:
            mot_in = video_motion_feat.float().contiguous().view(B * N, Dv)
        else:
            mot_in = ag.ops.prep_features_gather(video_motion_feat, rows, 1, False, False, err=err, out_dtype=torch.float32)
        mot = ag.linear(mot_in, self.visual_motion_input_unit.weight, self.visual_motion_input_unit.bias).view(B, N, D)
        visual, aq_embed, mq_embed, com_app, com_motion, aq_fusion, mq_fusion = self.visual_input_unit(
            app, mot, dynamic_q, words, qlen)
        pooled = self.feature_aggregation(visual)
        out = self.output_unit(question_embedding, pooled)
        return out, aq_embed, mq_embed, com_app, com_motion, aq_fusion, mq_fusion

    def forward(self, video_appearance_feat, video_motion_feat, question, question_len):
        """
        video_appearance_feat [B, N, F, vision_dim] fp32, video_motion_feat [B, N, vision_dim] fp32,
        question [B, L] int64, question_len [B] int64
        -> (logits [B, A] fp32, aq_embed, mq_embed [B,N,D], com_app[U], com_motion[U], aq_fusion[U], mq_fusion[U])
        """
        if not video_appearance_feat.is_cuda:
            raise RuntimeError("dualvgr_b200: DualVGR runs on sm_100a CUDA devices only; there is no CPU path")
        return self._forward(video_appearance_feat, video_motion_feat, question, question_len)

    def forward_from_store(self, dstore, rows, question, question_len):
        """forward() on the batch (dstore.app[rows], dstore.mot[rows]) of a device-resident feature store
        (loader.DeviceFeatureStore), read inside the two input prologue kernels: no batch of clip features is copied.
        rows [B] int32 on the store's device. Same returns as forward(), bit for bit. A row outside [0, V) reads zeros and
        sets dstore.err."""
        if not rows.is_cuda:
            raise RuntimeError("dualvgr_b200: DualVGR runs on sm_100a CUDA devices only; there is no CPU path")
        return self._forward(dstore.app, dstore.mot, question, question_len, rows, dstore.err)

    def _forward(self, video_appearance_feat, video_motion_feat, question, question_len, rows=None, err=None):
        """Body of forward() / forward_from_store(): only the two input prologues differ (rows None: dense batches)."""
        if ag.ACT[0] == torch.float32:
            return self._forward_fp32(video_appearance_feat, video_motion_feat, question, question_len, rows, err)
        ag.begin_forward()
        dev = video_appearance_feat.device
        N = video_motion_feat.shape[1]
        B = video_motion_feat.shape[0] if rows is None else rows.numel()
        D = self.visual_motion_input_unit.out_features
        qlen = question_len.to(torch.int32)
        # question encoder on a (high-priority) side stream: two 20-step recurrences over 256 sequences keep ~1/3 of the SMs
        # busy at most, so they run next to the appearance prologue / encoder instead of in front of them (the LSTM
        # kernels claim their tiles dynamically: sharing the GPU cannot stall them). Autograd runs the backward of a node on
        # the stream of its forward, so the question encoder's backward overlaps the appearance encoder's the same way.
        cur = torch.cuda.current_stream()
        side = fs.side_stream(dev, "question")
        side.wait_stream(cur)
        with torch.cuda.stream(side):
            launched = self.linguistic_input_unit.launch(question, qlen)       # kernels out first, autograd node last (below)
            # the question side of the Query Punishment Module of every unit layer only needs the question encoder: its
            # kernels go out right behind it, on the same stream, under the appearance encoder's recurrence
            chain = self.visual_input_unit.launch_query_chain(launched[1])
        # the two clip streams are carried as ONE stacked [2, B*N, D] tensor: both encoders write into its halves
        x0 = torch.empty((2, B * N, D), dtype=BF16, device=dev)
        app = self.visual_appearance_input_unit(video_appearance_feat, out=x0[0], rows=rows, err=err)
        if rows is None:
            mf = video_motion_feat if video_motion_feat.dtype == torch.bfloat16 else video_motion_feat.float()
            mot_in = ag.ops.prep_features(mf.contiguous().view(B * N, -1), 1, False, False)
        else:
            mot_in = ag.ops.prep_features_gather(video_motion_feat, rows, 1, False, False, err=err)
        mot = ag.linear(mot_in, self.visual_motion_input_unit.weight, self.visual_motion_input_unit.bias, out=x0[1]).view(B, N, D)
        with torch.cuda.stream(side):
            question_embedding, word_embedding, dynamic_q = self.linguistic_input_unit.fused(question, qlen, launched)
            query_all = self.visual_input_unit.query_chain(dynamic_q, word_embedding, qlen, chain)
        # (no join here: the unit stack waits for each layer's queries through the chain's per-layer events, and the main
        #  stream only needs the question embedding at the classifier)
        for t in (question_embedding, word_embedding, dynamic_q, query_all):
            t.record_stream(cur)
        hook = getattr(self, "_unit_inputs_grad_hook", None)
        if hook is not None and torch.is_grad_enabled():
            # data-parallel engine: tell it when the gradients of everything DOWNSTREAM of the three encoders are final, so
            # that their all-reduce overlaps the encoders' backward (engine.TrainEngine)
            hooked = [t for t in (app, mot, dynamic_q, word_embedding) if t.requires_grad]
            hook.arm(len(hooked))
            for t in hooked:
                t.register_hook(hook)
        visual, aq_embed, mq_embed, com_app, com_motion, aq_fusion, mq_fusion = self.visual_input_unit.fused(
            app, mot, dynamic_q, word_embedding, qlen, query_all=query_all, chain=chain)
        pooled = self.feature_aggregation(visual)
        cur.wait_stream(side)
        out = self.output_unit(question_embedding, pooled)
        return out, aq_embed, mq_embed, com_app, com_motion, aq_fusion, mq_fusion


class DualVGRUnit_multiple(nn.Module):
    def __init__(self, word_dim=300, module_dim=512, num_of_nodes=8, appearance_graph_layers=1, motion_graph_layers=1,
                 graph_module='GAT', unit_layers=3):
        super().__init__()
        if appearance_graph_layers != 1 or motion_graph_layers != 1:
            raise NotImplementedError("graph_layers must be 1 (every shipped config; for >1 the reference aliases layers "
                                      "through its [i+j] indexing, model/models.py:151-158)")
        self.layers = unit_layers
        self.word_dim = word_dim
        self.queryAttn = nn.ModuleList([QueryAttn(module_dim=module_dim) for _ in range(unit_layers)])
        self.queryPunish_appear = nn.ModuleList([QueryPunish(word_dim=word_dim, module_dim=module_dim) for _ in range(unit_layers)])
        self.queryPunish_motion = nn.ModuleList([QueryPunish(word_dim=word_dim, module_dim=module_dim) for _ in range(unit_layers)])
        if graph_module == 'GAT':
            mk = lambda: nn.ModuleList([punishGAT(module_dim, module_dim // 4, dropout=0.15, alpha=0.01, n_heads=4)
                                        for _ in range(unit_layers)])
            self.appearance_GCN = mk()
            self.motion_GCN = mk()
            self.acGCN = mk()
            self.mcGCN = mk()
        elif unit_layers > 0:
            raise NotImplementedError("only graph_module='GAT' builds graph layers (reference model/models.py:94)")
        self.attention_appearance = nn.ModuleList([AttentionSFGCN(module_dim, module_dim) for _ in range(unit_layers)])
        self.attention_motion = nn.ModuleList([AttentionSFGCN(module_dim, module_dim) for _ in range(unit_layers)])
        self.num_of_appearance_graph_layers = appearance_graph_layers
        self.num_of_motion_graph_layers = motion_graph_layers
        self.visualfusion = MFB([module_dim, module_dim], module_dim)
        self.module_dim = module_dim
        self.activation = nn.ELU()
        adj = build_adjacency(num_of_nodes)
        self.register_buffer("appearance_adj", adj.clone(), persistent=False)
        self.register_buffer("motion_adj", adj.clone(), persistent=False)

    def _query_params(self):
        return [p for i in range(self.layers) for p in fs.unit_layer_params(self, i)[:8]]

    def launch_query_chain(self, question_state):
        """Launches the forward kernels of fused_stack.QueryChainFn on the current stream from the question encoder's raw
        launch state (fused_stack.QuestionInputFn.launch) — no autograd node yet; query_chain() adopts the result."""
        if self.layers == 0:
            return None
        B, L, W, Wp, H = question_state["cfg"][:5]
        dq = question_state["seq_out"].view(B * L, 4 * H)[:, :2 * H]
        qlen = question_state["qlen"]
        return fs.QueryChainFn.launch(self.word_dim, dq, question_state["words"], qlen, self._query_params())

    def query_chain(self, dq2, words_p, qlen, launched=None):
        """The cycle queries of every layer, [U, B, 2D] bf16 (fused_stack.QueryChainFn)."""
        if self.layers == 0:
            return torch.zeros((0, words_p.shape[0], 2 * self.module_dim), dtype=BF16, device=words_p.device)
        return fs.QueryChainFn.apply((self.word_dim, launched), dq2, words_p, qlen, *self._query_params())

    def fused(self, app, mot, dq2, words_p, qlen, query_all=None, chain=None):
        """The whole stack as ONE autograd Function (fused_stack.UnitStackFn): app / mot [B,N,D] bf16, dq2 [B*L, D] bf16
        (row stride free), words_p [B,L,Wp] bf16 zero-padded, qlen int32. Same returns as forward()."""
        U = self.layers
        if query_all is None:
            query_all = self.query_chain(dq2, words_p, qlen)
        heads = self.acGCN[0].n_heads if U > 0 else 4
        pdrop = self.acGCN[0].dropout if (U > 0 and self.training) else 0.0
        params = [p for i in range(U) for p in fs.unit_layer_params(self, i)]
        grad = torch.is_grad_enabled()
        if chain is None and grad and query_all.grad_fn is not None:
            chain = getattr(query_all.grad_fn, "pre", None)
        cfg = (U, heads, float(pdrop), self.word_dim, getattr(self, "_aux", None) if grad else None, grad, chain)
        outs = fs.UnitStackFn.apply(cfg, app, mot, query_all, self.appearance_adj, *params)
        app, mot, aq_embed, mq_embed = outs[:4]
        f32 = outs[4:]
        com_app_list = [f32[4 * i] for i in range(U)]
        aq_fusion_list = [f32[4 * i + 1] for i in range(U)]
        com_motion_list = [f32[4 * i + 2] for i in range(U)]
        mq_fusion_list = [f32[4 * i + 3] for i in range(U)]
        visual = self.visualfusion([app, mot])
        return visual, aq_embed, mq_embed, com_app_list, com_motion_list, aq_fusion_list, mq_fusion_list

    def forward(self, appearance_video_feat, motion_video_feat, dynamic_question_embedding, word_embedding, question_len):
        """app / motion [B,N,D], dynamic_q [B,L,D], words [B,L,W], question_len [B] ->
        (visual [B,N,D], aq_embed, mq_embed, com_app[U], com_motion[U], aq_fusion[U], mq_fusion[U])
        Module-by-module path (one autograd Function per mirrored module); DualVGR.forward uses fused()."""
        B, N, D = appearance_video_feat.shape
        app = appearance_video_feat.to(ag.ACT[0])
        mot = motion_video_feat.to(ag.ACT[0])
        dq = dynamic_question_embedding.to(ag.ACT[0])
        words = pad_last(word_embedding).to(ag.ACT[0])
        qlen = question_len.to(torch.int32)
        adj = self.appearance_adj
        aq_fusion_list, mq_fusion_list, com_app_list, com_motion_list = [], [], [], []
        aq_embed = mq_embed = None
        for i in range(self.layers):
            # Query Punishment Module: word attention -> cycle query -> per-clip gates of both streams
            q_c, _ = self.queryAttn[i](words, dq, qlen, word_dim=self.word_dim)
            qa, qm = self.queryPunish_appear[i].query_weight, self.queryPunish_motion[i].query_weight
            query = ag.linear_cat(q_c, qa.weight, qa.bias, qm.weight, qm.bias)      # [B, 2D]: both streams' queries, one GEMM
            g_app, g_mot = ag.GateFn.apply(app, mot, query)
            # multi-view GAT: common + specific graph of each stream, one fused launch for the four graphs
            (z_app, z_mot), (com_app, aq_fusion, com_mot, mq_fusion) = fused_gat_layer(
                [self.acGCN[i], self.appearance_GCN[i], self.mcGCN[i], self.motion_GCN[i]], [0, 0, 1, 1],
                [app, mot], [g_app, g_mot], adj, self.training)
            aq_fusion_list.append(aq_fusion); com_app_list.append(com_app)
            mq_fusion_list.append(mq_fusion); com_motion_list.append(com_mot)
            # common-vs-specific view attention + residual
            app, aq_embed = self.attention_appearance[i].fused(z_app, app)
            mot, mq_embed = self.attention_motion[i].fused(z_mot, mot)
        visual = self.visualfusion([app, mot])
        return visual, aq_embed, mq_embed, com_app_list, com_motion_list, aq_fusion_list, mq_fusion_list
