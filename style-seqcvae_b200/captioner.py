"""Drop-in `UpDownCaptioner` for the reference's var_updown model, running on libsscvae_b200.so.

Mirrors var_updown/var_updown/models/updown_captioner.py:20-466 of visinf/style-seqcvae: same ctor and
`from_config` arguments, same `forward` signature and outputs (training: {"loss": (B,), "kld": (B,)};
otherwise {"predictions": (B, steps)} int64), same `state_dict` keys and shapes, so reference
checkpoints load and `train.py` / `inference.py` work unchanged (INTEGRATION.md).

The nn.Module below owns nothing but parameters: the torch sub-modules are parameter containers whose
`forward` is never called. All arithmetic of the hot path (the T-step UpDown cell, latent nets, KL/CE,
BPTT, beam/CBS search) happens in hand-written sm_100a kernels behind the C ABI; there is no eager /
CPU fallback — without a CUDA device and the built library this module raises.
"""
import ctypes as C
import weakref
from typing import Dict, Optional

import torch
from torch import nn
from torch.utils.weak import WeakIdKeyDictionary

from . import _lib

# weight tensor -> weak reference to the captioner whose packed operands were last built from it: FusedClipSGD finds the
# captioner of its parameters here and updates the packed operands together with the weights
PACKED_OWNERS = WeakIdKeyDictionary()


class _ButdAttentionParams(nn.Module):
    """Parameter container with the reference's names (updown-baseline/updown/modules/attention.py:27-34)."""

    def __init__(self, query_size, image_feature_size, projection_size):
        super().__init__()
        self._query_vector_projection_layer = nn.Linear(query_size, projection_size, bias=False)
        self._image_features_projection_layer = nn.Linear(image_feature_size, projection_size, bias=False)
        self._attention_layer = nn.Linear(projection_size, 1, bias=False)


class _UpDownCellParams(nn.Module):
    """Parameter container with the reference's names and shapes
    (var_updown/var_updown/modules/updown_cell.py:34-84)."""

    def __init__(self, F, E, H, A, Z, cond):
        super().__init__()
        self._attention_lstm_cell = nn.LSTMCell(E + F + 2 * H, H)
        self._butd_attention = _ButdAttentionParams(H, F, A)
        self._language_lstm_cell_encoder = nn.LSTMCell(cond + F + 2 * H, H)
        self._language_lstm_cell_decoder = nn.LSTMCell(cond + F + 2 * H + Z, H)
        self.fc_mean = nn.Linear(H, Z)
        self.fc_log_var = nn.Linear(H, Z)


class _TrainStep(torch.autograd.Function):
    """forward = sscvae_train_forward, backward = sscvae_train_backward (BPTT kernels)."""

    @staticmethod
    def forward(ctx, module, image_features, caption_tokens, sentiment, obj_means, eps, seed, *params):
        L = _lib.lib()
        B, N, _ = image_features.shape
        packed = module._packed_weights()
        ws = module._train_workspace(B, N)
        # The library replays a call as a CUDA graph when it sees the same pointers again, so everything the call reads
        # or writes lives at stable addresses: the per-row losses (and, in backward, their incoming gradients) go through
        # four small persistent buffers instead of fresh allocator blocks, whose addresses are not guaranteed to repeat
        # (observed: sporadic re-captures inside the timed region, 7.4 -> 10-11.7 ms per end-to-end step).
        loss_buf, kld_buf, _, _ = module._io_buffers(B, image_features.device)
        stream = C.c_void_p(torch.cuda.current_stream(image_features.device).cuda_stream)
        wptr = _lib.ptr_array(module._weight_tensors())
        _lib.check(L.sscvae_train_forward(
            module._handle, B, N, _lib.ptr(packed), wptr, _lib.ptr(image_features), _lib.ptr(caption_tokens),
            _lib.ptr(sentiment), _lib.ptr(obj_means), _lib.ptr(eps), C.c_uint64(seed), _lib.ptr(ws), ws.numel(), _lib.ptr(loss_buf),
            _lib.ptr(kld_buf), stream))
        module._ws_generation += 1
        ctx.module, ctx.B, ctx.N, ctx.generation = module, B, N, module._ws_generation
        ctx.keep = (image_features, caption_tokens, sentiment, obj_means, eps)
        return loss_buf.clone(), kld_buf.clone()

    @staticmethod
    def backward(ctx, grad_loss, grad_kld):
        module = ctx.module
        if ctx.generation != module._ws_generation:
            raise RuntimeError("sscvae: backward() after a newer forward() reused the training workspace; "
                               "call backward before the next forward")
        L = _lib.lib()
        params = module._weight_tensors()
        needs = ctx.needs_input_grad[7:]
        # Gradients are written into persistent per-bucket flat buffers (stable pointers: the backward graph is replayed,
        # and the data-parallel all-reduce runs in place on the buckets). If a parameter still holds the previous
        # gradient in that very storage (gradient accumulation without zero_grad), a fresh tensor is used instead.
        views = module._grad_views()
        grads = []
        for p, need, v in zip(params, needs, views):
            if not (need and p.requires_grad) or v is None:
                grads.append(None)
            elif p.grad is not None and p.grad.data_ptr() == v.data_ptr():
                grads.append(torch.empty_like(p))
            else:
                grads.append(v)
        dev = grad_loss.device
        _, _, gl, gk = module._io_buffers(ctx.B, dev)
        if grad_loss is not None:
            gl.copy_(grad_loss)
        else:
            gl.zero_()
        if grad_kld is not None:
            gk.copy_(grad_kld)
        else:
            gk.zero_()
        ws = module._train_workspace(ctx.B, ctx.N)
        stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        events = module._group_events
        ev = None
        if events is not None:
            # torch creates the underlying cudaEvent_t lazily, at the first record(): an event that was never recorded has
            # handle 0, the library would skip its record and a later wait_event() on it would be a no-op (the all-reduce
            # would then race with the backward kernels). Force creation here; the library re-records them.
            for e in events:
                if not e.cuda_event:
                    e.record(torch.cuda.current_stream(dev))
            handles = [e.cuda_event for e in events]
            if len(handles) != _lib.GRAD_GROUPS or not all(handles):
                raise RuntimeError("sscvae: gradient-bucket events must be %d created CUDA events" % _lib.GRAD_GROUPS)
            ev = (C.c_void_p * _lib.GRAD_GROUPS)(*handles)
        _lib.check(L.sscvae_train_backward(
            module._handle, ctx.B, ctx.N, _lib.ptr(module._packed_weights()), _lib.ptr_array(params), _lib.ptr(ws),
            ws.numel(), _lib.ptr(gl), _lib.ptr(gk), _lib.ptr_array(grads), ev, stream))
        # A gradient that was written into the bucket view becomes `.grad` directly (autograd's AccumulateGrad would
        # clone a tensor that somebody else still references, and the in-place all-reduce of the buckets relies on
        # p.grad being the view itself); anything else goes through autograd's normal accumulation.
        out = []
        for p, g, v in zip(params, grads, views):
            if g is not None and g is v and p.grad is None:
                p.grad = v
                out.append(None)
            else:
                out.append(g)
        return (None, None, None, None, None, None, None) + tuple(out)


class _TrainDecodeStep(torch.autograd.Function):
    """One training step of the cell: forward = sscvae_train_step_forward, backward = sscvae_train_step_backward.

    Inputs: module, boxes N, image state (uint8), sentiment, prev tokens, eps, seed, tape (uint8), the six input states (or
    Nones), then the parameters. Outputs: logits, the six states, mean, log_var, prior mean (sentiment_vae == 2, else
    empty), alpha."""

    @staticmethod
    def forward(ctx, module, N, state, sentiment, prev, eps, seed, tape, *rest):
        states, params = rest[:6], rest[6:]
        outs = module._train_step_call(N, state, sentiment, prev, None if states[0] is None else states, eps, seed, tape)
        ctx.module, ctx.state, ctx.tape, ctx.shape = module, state, tape, (prev.numel(), N)
        ctx.has_states = states[0] is not None
        # the parameters are saved so that an in-place update before backward raises autograd's version error
        ctx.save_for_backward(*params)
        if outs[9].numel() == 0:
            ctx.mark_non_differentiable(outs[9])
        ctx.set_materialize_grads(False)
        return outs

    @staticmethod
    def backward(ctx, d_logits, *d):
        module = ctx.module
        params = ctx.saved_tensors                       # raises if a parameter was modified in place since forward
        d_states, d_mean, d_log_var, d_pm, d_alpha = d[:6], d[6], d[7], d[8], d[9]
        B, N = ctx.shape
        dev = params[0].device
        if d_logits is None:
            d_logits = torch.zeros(B, module._vocab_size, device=dev)
        f = lambda t: None if t is None or t.numel() == 0 else t.contiguous().float()
        # held in locals until the call has been enqueued: a temporary's block could otherwise be handed to the next one
        d_logits, d_mean, d_log_var, d_pm, d_alpha = f(d_logits), f(d_mean), f(d_log_var), f(d_pm), f(d_alpha)
        d_states = [f(t) for t in d_states]
        n_in = 8
        needs = ctx.needs_input_grad
        d_in = [torch.empty(B, module.hidden_size, device=dev) if ctx.has_states and needs[n_in + k] else None
                for k in range(6)]
        grads = []
        for i, p in enumerate(params):
            want = needs[n_in + 6 + i] and not (module._tied and i == 0)
            grads.append(torch.empty_like(p) if want else None)
        L = _lib.lib()
        ws = module._train_step_workspace(B, N)
        stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        _lib.check(L.sscvae_train_step_backward(
            module._handle, B, N, _lib.ptr(module._packed_weights()), _lib.ptr_array(params), _lib.ptr(ctx.state),
            ctx.state.numel(), _lib.ptr(ctx.tape), ctx.tape.numel(), _lib.ptr(ws), ws.numel(), _lib.ptr(d_logits),
            _lib.ptr_array(d_states), _lib.ptr(d_mean), _lib.ptr(d_log_var), _lib.ptr(d_pm), _lib.ptr(d_alpha),
            _lib.ptr_array(d_in), _lib.ptr_array(grads), stream))
        return (None,) * n_in + tuple(d_in) + tuple(grads)


class UpDownCaptioner(nn.Module):
    def __init__(
        self,
        vocabulary,
        image_feature_size,
        embedding_size,
        hidden_size,
        attention_projection_size,
        max_caption_length=20,
        beam_size=1,
        use_cbs=False,
        min_constraints_to_satisfy=2,
        z_space=150,
        prior_std=None,
        simple_vae=False,
        latent_embedding=None,
        latent_embedding_multip=1,
        sentiment_vae=False,
        senti_prior_multip=1,
        cbs_simple=False,
        device=None,
        glove_vectors: Optional[torch.Tensor] = None,
        mean_choice: Optional[dict] = None,
    ):
        super().__init__()
        self._vocabulary = vocabulary
        self.image_feature_size = image_feature_size
        self.embedding_size = embedding_size
        self.hidden_size = hidden_size
        self.attention_projection_size = attention_projection_size
        self._max_caption_length = max_caption_length
        self._use_cbs = use_cbs
        self._min_constraints_to_satisfy = min_constraints_to_satisfy
        self.z_space = z_space
        _vocab_size = vocabulary.get_vocab_size()
        self._vocab_size = _vocab_size
        self._pad_index = vocabulary.get_token_index("@@UNKNOWN@@")
        self._boundary_index = vocabulary.get_token_index("@@BOUNDARY@@")
        self.prior_std = 1.0 if prior_std is None else prior_std
        self.sentiment_vae = int(sentiment_vae)
        self.senti_prior_multip = senti_prior_multip
        self.simple_vae = bool(simple_vae)
        self.latent_embedding = latent_embedding
        self.latent_embedding_multip = latent_embedding_multip
        self.beam_size = beam_size
        self.per_node_beam_size = (beam_size // 2) or beam_size     # updown_captioner.py:134, cbs.py:57
        self.device = device
        self.cbs_simple = cbs_simple
        if self.sentiment_vae not in (0, 1, 2):
            raise NotImplementedError()                              # updown_cell.py:72-73
        if latent_embedding not in ("glove", "senti_word_net"):
            raise NotImplementedError()                              # updown_cell.py:169-174
        # sentiment_vae == 2: {attribute word: (Z,) vector} the per-box attribute means are built from. The reference loads
        # it from hard-coded pickle / json paths in its ctor (updown_captioner.py:76-93); here it is an argument (and forward()
        # also accepts the already translated (B, N, Z) tensor).
        self.mean_choice = mean_choice

        self._tied = embedding_size in (300, 600)                    # updown_captioner.py:75
        if self._tied:
            if glove_vectors is None:
                # the reference's rule for words without a pre-trained vector (updown_captioner.py:197,209,215)
                glove_vectors = 2 * torch.randn(_vocab_size, embedding_size) - 1
                glove_vectors[self._pad_index] = 0
            self._embedding_layer = nn.Embedding.from_pretrained(glove_vectors, freeze=True, padding_idx=self._pad_index)
        else:
            self._embedding_layer = nn.Embedding(_vocab_size, embedding_size, padding_idx=self._pad_index)
            assert not use_cbs, "CBS is not supported without Frozen GloVe embeddings (300d / 600d)"

        # width of the conditioning block of the encoder / decoder LSTM inputs (updown_cell.py:47-81; the reference writes
        # the "glove" width of sentiment_vae == 2 as the literal 150 = its Z_SPACE)
        if self.simple_vae or self.sentiment_vae == 0:
            cond = 0
        elif self.sentiment_vae == 1 or latent_embedding == "senti_word_net":
            cond = 1
        else:
            cond = z_space
        self._updown_cell = _UpDownCellParams(image_feature_size, embedding_size, hidden_size,
                                              attention_projection_size, z_space, cond)
        if self._tied:
            self._output_projection = nn.Sequential(nn.Linear(hidden_size, embedding_size), nn.Tanh())
            self._output_layer = nn.Linear(embedding_size, _vocab_size, bias=False)
            self._output_layer.weight = self._embedding_layer.weight
        else:
            self._output_projection = nn.Identity()
            self._output_layer = nn.Linear(hidden_size, _vocab_size)

        # ---- native state (not part of state_dict)
        dims = _lib.SscvaeDims(
            image_feature_size, embedding_size, hidden_size, attention_projection_size, z_space, _vocab_size,
            max_caption_length, self.sentiment_vae, int(self.simple_vae), int(self._tied), self._pad_index,
            self._boundary_index, float(self.prior_std), float(senti_prior_multip),
            int(latent_embedding == "senti_word_net"))
        self._dims = dims
        self._handle = C.c_void_p()
        _lib.check(_lib.lib().sscvae_create(C.byref(dims), C.byref(self._handle)))
        self._packed = None
        self._packed_key = None
        self._ws_cache: Dict[tuple, torch.Tensor] = {}
        self._ws_generation = 0
        self._group_events = None          # set by the data-parallel wrapper
        self._grad_view_cache = None
        self._grad_flat = {}
        self.rng_mode = "philox"           # "reference": draw eps from the CPU generator like updown_cell.py:206
        # True: outputs also carry "attention", the attention weights over the boxes behind every word (the last element
        # of the reference's eval step, updown_captioner.py:371-455): fp32, new tensors, not differentiable
        self.return_attention = False
        # True: _decode_step also runs in training mode, as the reference's training loop calls it (updown_captioner.py:282-310):
        # a differentiable step per call, for per-step objectives; the fused training forward() stays the fast path
        self.stepwise_training = False
        self._eps_override = None          # tests: explicit eps tensor
        self._call_counter = 0
        self.last_search = None

    def __del__(self):
        try:
            if getattr(self, "_handle", None):
                _lib.lib().sscvae_destroy(self._handle)
                self._handle = None
        except Exception:
            pass

    @classmethod
    def from_config(cls, config, **kwargs):
        _C = config
        vocabulary = kwargs.pop("vocabulary")
        return cls(
            vocabulary=vocabulary,
            image_feature_size=_C.MODEL.IMAGE_FEATURE_SIZE,
            embedding_size=_C.MODEL.EMBEDDING_SIZE,
            hidden_size=_C.MODEL.HIDDEN_SIZE,
            attention_projection_size=_C.MODEL.ATTENTION_PROJECTION_SIZE,
            beam_size=_C.MODEL.BEAM_SIZE,
            max_caption_length=_C.DATA.MAX_CAPTION_LENGTH,
            use_cbs=_C.MODEL.USE_CBS,
            min_constraints_to_satisfy=_C.MODEL.MIN_CONSTRAINTS_TO_SATISFY,
            z_space=_C.MODEL.Z_SPACE,
            prior_std=_C.MODEL.PRIOR_STD,
            simple_vae=_C.MODEL.SIMPLE_VAE,
            latent_embedding=_C.MODEL.LATENT_EMBEDDING,
            sentiment_vae=_C.MODEL.SENTIMENT_VAE,
            senti_prior_multip=_C.MODEL.SENTI_PRIOR_MULTIP,
            latent_embedding_multip=_C.MODEL.LATENT_EMBEDDING_MULTIP,
            cbs_simple=_C.MODEL.CBS_SIMPLE,
            device=kwargs["device"],
        )

    # ------------------------------------------------------------------------------------------
    def _weight_tensors(self):
        """Parameters in SSCVAE_W_* order (include/sscvae.h)."""
        c = self._updown_cell
        out = [self._embedding_layer.weight]
        for cell in (c._attention_lstm_cell,):
            out += [cell.weight_ih, cell.weight_hh, cell.bias_ih, cell.bias_hh]
        a = c._butd_attention
        out += [a._query_vector_projection_layer.weight, a._image_features_projection_layer.weight, a._attention_layer.weight]
        for cell in (c._language_lstm_cell_encoder, c._language_lstm_cell_decoder):
            out += [cell.weight_ih, cell.weight_hh, cell.bias_ih, cell.bias_hh]
        out += [c.fc_mean.weight, c.fc_mean.bias, c.fc_log_var.weight, c.fc_log_var.bias]
        if self._tied:
            out += [self._output_projection[0].weight, self._output_projection[0].bias]
        else:
            out += [self._output_layer.weight, self._output_layer.bias]
        return out

    def _require_cuda(self, t: torch.Tensor):
        if not t.is_cuda:
            raise RuntimeError("sscvae UpDownCaptioner runs only on a CUDA (sm_100a) device: move the module and its "
                               "inputs to cuda; there is no CPU fallback")
        for p in self._weight_tensors():
            if p.device != t.device or p.dtype != torch.float32 or not p.is_contiguous():
                raise RuntimeError("sscvae: parameters must be contiguous fp32 tensors on the input's device")

    def _features(self, image_features: torch.Tensor) -> torch.Tensor:
        """fp32 (the reference's format) or bf16 region features (the bf16 feature cache, `sscvae.pack_features`): bf16
        inputs are consumed as they are - half the host->device bytes, bit-identical results - anything else is
        converted to fp32. Tells the library which of the two the following call gets."""
        if image_features.dtype == torch.bfloat16:
            image_features = image_features.contiguous()
        else:
            image_features = image_features.contiguous().float()
        _lib.check(_lib.lib().sscvae_set_option(self._handle, b"features_bf16", int(image_features.dtype == torch.bfloat16)))
        return image_features

    def _reuse_image_state(self, ws_key, image_features) -> None:
        """Decode calls on the SAME feature tensor (the reference's loop over latent samples) reuse the per-image state
        left in the decode workspace by the previous call: the analogue of the reference's lru_cache on the projected
        features (attention.py:99), keyed like it on tensor identity. The previous tensor is kept alive here, so a new
        tensor can never alias its storage; an in-place update bumps the version counter; new weights or another
        workspace invalidate the state as well."""
        key = (ws_key, image_features._version, tuple(image_features.shape), image_features.dtype,
               tuple((p.data_ptr(), p._version) for p in self._weight_tensors()))
        last = getattr(self, "_image_state", None)
        reuse = last is not None and last[0] is image_features and last[1] == key
        self._image_state = (image_features, key)
        _lib.check(_lib.lib().sscvae_set_option(self._handle, b"reuse_image_state", int(reuse)))

    def _packed_weights(self) -> torch.Tensor:
        ws = self._weight_tensors()
        # one key per weight: a weight is re-packed when its storage or its version counter changed (torch's own
        # optimizers bump the counter; FusedClipSGD, which writes through raw pointers, does so explicitly)
        key = self._weights_key(ws)
        if self._packed is None or key != self._packed_key or self._packed.device != ws[0].device:
            L = _lib.lib()
            nbytes = L.sscvae_packed_bytes(self._handle)
            dirty = None
            if self._packed is None or self._packed.numel() != nbytes or self._packed.device != ws[0].device:
                self._packed = torch.empty(nbytes, dtype=torch.uint8, device=ws[0].device)
            elif self._packed_key is not None:
                dirty = (C.c_uint8 * len(ws))(*[int(a != b) for a, b in zip(key, self._packed_key)])
            stream = C.c_void_p(torch.cuda.current_stream(ws[0].device).cuda_stream)
            _lib.check(L.sscvae_pack_weights(self._handle, _lib.ptr_array(ws), _lib.ptr(self._packed), nbytes, dirty,
                                             stream))
            self._packed_key = key
            me = weakref.ref(self)
            for p in ws:
                PACKED_OWNERS[p] = me
        return self._packed

    @staticmethod
    def _weights_key(ws) -> tuple:
        return tuple((p.data_ptr(), p._version) for p in ws)

    def _sgd_step_packed(self, ps, grads, bufs, firsts, hyper, scratch) -> bool:
        """FusedClipSGD.step() for parameters `ps` of this module: the update and the re-pack of their bf16 / fp32
        images in the packed operands in one pass (sscvae_sgd_step_packed), so the next forward re-packs nothing.
        Returns False, having done nothing, unless the packed operands are current (built from exactly these
        weights, none changed since), every tensor of `ps` is one of the weights, and the weights are contiguous fp32
        tensors on the device of the packed operands. `hyper`: max_norm, lr, momentum, weight_decay, grad_scale."""
        ws = self._weight_tensors()
        if self._packed is None or self._packed_key != self._weights_key(ws):
            return False
        dev = self._packed.device
        if any(w.device != dev or w.dtype != torch.float32 or not w.is_contiguous() for w in ws):
            return False
        slot = {id(w): i for i, w in enumerate(ws)}
        order = [slot.get(id(p)) for p in ps]
        if None in order or len(set(order)) != len(order):
            return False
        n = len(ws)
        g_by_id, b_by_id, f_by_id = [None] * n, [None] * n, [0] * n
        for i, g, b, f in zip(order, grads, bufs, firsts):
            g_by_id[i], b_by_id[i], f_by_id[i] = g, b, f
        L = _lib.lib()
        stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        _lib.check(L.sscvae_sgd_step_packed(
            self._handle, _lib.ptr_array(ws), _lib.ptr_array(g_by_id), _lib.ptr_array(b_by_id),
            (C.c_int32 * n)(*f_by_id), len(order), (C.c_int32 * len(order))(*order), *[float(h) for h in hyper],
            _lib.ptr(self._packed), self._packed.numel(), _lib.ptr(scratch), scratch.numel(), stream))
        for p in ps:
            torch.autograd.graph.increment_version(p)
        self._packed_key = self._weights_key(ws)      # the packed operands already hold the updated weights
        return True

    def _grad_views(self):
        """Per weight tensor (SSCVAE_W_* order): a view, shaped like the parameter, into the flat gradient buffer of its
        data-parallel bucket (dp.GROUP_PREFIXES)."""
        ws = self._weight_tensors()
        dev = ws[0].device
        if self._grad_view_cache is not None and self._grad_view_cache[0] == dev:
            return self._grad_view_cache[1]
        from .dp import group_of, GROUP_PREFIXES
        names = {id(p): n for n, p in self.named_parameters()}
        groups = [[] for _ in GROUP_PREFIXES]
        for i, p in enumerate(ws):
            n = names.get(id(p))
            if n is not None:                      # every parameter, also currently frozen ones (train.py:156-161 toggles)
                groups[group_of(n)].append(i)
        views = [None] * len(ws)
        self._grad_flat = {}
        for g, idxs in enumerate(groups):
            if not idxs:
                continue
            flat = torch.zeros(sum(ws[i].numel() for i in idxs), dtype=torch.float32, device=dev)
            off = 0
            for i in idxs:
                views[i] = flat[off:off + ws[i].numel()].view_as(ws[i])
                off += ws[i].numel()
            self._grad_flat[g] = (flat, [(ws[i], views[i]) for i in idxs])
        self._grad_view_cache = (dev, views)
        return views

    def grad_buckets(self):
        """{bucket: (flat fp32 buffer, [(parameter, view into the buffer), ...])} for an in-place gradient all-reduce."""
        self._grad_views()
        return self._grad_flat

    def _train_workspace(self, B, N) -> torch.Tensor:
        dev = self._embedding_layer.weight.device
        key = ("train", B, N, dev)
        ws = self._ws_cache.get(key)
        if ws is None:
            nbytes = _lib.lib().sscvae_train_workspace_bytes(self._handle, B, N)
            self._ws_cache = {k: v for k, v in self._ws_cache.items() if k[0] != "train"}
            ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
            self._ws_cache[key] = ws
        return ws

    def train_region(self, B, N, name, dtype, shape):
        """Typed view of a named region of the training workspace (tests / debugging)."""
        off, nb = C.c_size_t(), C.c_size_t()
        _lib.check(_lib.lib().sscvae_train_region(self._handle, B, N, name.encode(), C.byref(off), C.byref(nb)))
        ws = self._train_workspace(B, N)
        n = 1
        for s in shape:
            n *= s
        itemsize = torch.empty(0, dtype=dtype).element_size()
        assert n * itemsize <= nb.value, (name, n * itemsize, nb.value)
        return ws[off.value: off.value + n * itemsize].view(dtype).view(*shape)

    def decode_region(self, B, N, S, K, name, dtype, shape):
        """Typed view of a named region of the last decode workspace (tests / debugging)."""
        off, nb = C.c_size_t(), C.c_size_t()
        _lib.check(_lib.lib().sscvae_decode_region(self._handle, B, N, S, K, name.encode(), C.byref(off), C.byref(nb)))
        ws = self._ws_cache[("decode", B, N, S, K, self._embedding_layer.weight.device)]
        n = 1
        for s in shape:
            n *= s
        itemsize = torch.empty(0, dtype=dtype).element_size()
        assert n * itemsize <= nb.value, (name, n * itemsize, nb.value)
        return ws[off.value: off.value + n * itemsize].view(dtype).view(*shape)

    def _io_buffers(self, B, device):
        """(loss, kld, grad_loss, grad_kld): persistent (B,) fp32 buffers the C calls read and write (stable pointers)."""
        key = ("io", B, device)
        bufs = self._ws_cache.get(key)
        if bufs is None:
            bufs = tuple(torch.zeros(B, dtype=torch.float32, device=device) for _ in range(4))
            self._ws_cache[key] = bufs
        return bufs

    def _next_seed(self) -> int:
        """Philox seed of the next call: (torch seed, call counter, data-parallel rank). The rank term gives every
        replica its own noise stream even when all ranks call torch.manual_seed with the same value (SURVEY 8e:
        disjoint per-rank eps streams)."""
        self._call_counter += 1
        seed = (int(torch.initial_seed()) * 1000003 + self._call_counter) & 0xFFFFFFFFFFFFFFFF
        if torch.distributed.is_available() and torch.distributed.is_initialized():
            seed ^= ((torch.distributed.get_rank() + 1) * 0x9E3779B97F4A7C15) & 0xFFFFFFFFFFFFFFFF
        return seed

    # ------------------------------------------------------------------------------------------
    def forward(
        self,
        image_features: torch.Tensor,
        obj_atts=None,
        image_attributes=None,
        caption_tokens=None,
        sentiment=None,
        fsm: torch.Tensor = None,
        num_constraints: torch.Tensor = None,
        constraints=None,
        constraint2states=None,
    ):
        self._require_cuda(image_features)
        image_features = self._features(image_features)
        B, N, F = image_features.shape
        if F != self.image_feature_size:
            raise ValueError(f"image_features last dim {F} != image_feature_size {self.image_feature_size}")
        cond = self.sentiment_vae == 1
        if cond:
            if sentiment is None:
                raise ValueError("sentiment is required when sentiment_vae == 1")
            sentiment = sentiment.to(image_features.device).contiguous().float().view(B, 1)
        else:
            sentiment = None
        obj_means = self._obj_means(obj_atts, B, N, image_features.device)

        if self.training and caption_tokens is not None:
            caption_tokens = caption_tokens.to(image_features.device).contiguous().long()
            if caption_tokens.shape != (B, self._max_caption_length):
                raise ValueError(f"caption_tokens must be (B, {self._max_caption_length}), got {tuple(caption_tokens.shape)}")
            # nn.Embedding raises on an out-of-range id; the kernels index the table unchecked, so check on the device
            # (asynchronous: no host sync on the training path)
            torch._assert_async(((caption_tokens >= 0) & (caption_tokens < self._vocab_size)).all(),
                                "caption_tokens contains an id outside [0, vocab_size)")
            T = self._max_caption_length + 1
            eps = self._eps_override
            if eps is None and self.rng_mode == "reference":
                # one (B,Z) CPU draw per step, in step order, exactly like updown_cell.py:206
                eps = torch.stack([torch.randn(B, self.z_space) for _ in range(T)]).to(image_features.device)
            if eps is not None:
                eps = eps.to(image_features.device).contiguous().float()
                assert eps.shape == (T, B, self.z_space)
            loss, kld = _TrainStep.apply(self, image_features, caption_tokens, sentiment, obj_means, eps, self._next_seed(),
                                         *self._weight_tensors())
            out = {"loss": loss, "kld": kld}
            if self.return_attention:
                # the forward kernels keep alpha time-major, (T, B, N), for the backward pass: a (B, T, N) copy
                alpha = self.train_region(B, N, "alpha", torch.float32, (T, B, N))
                out["attention"] = alpha.detach().transpose(0, 1).clone(memory_format=torch.contiguous_format)
            return out

        pred, attention = self._decode(image_features, sentiment, fsm, num_constraints, obj_means, constraints,
                                       constraint2states)
        out = {"predictions": pred}
        if attention is not None:
            out["attention"] = attention
        return out

    def _decode_attention(self, ws, valid, num_boxes, rows, all_shape=None):
        """sscvae_decode_attention on the workspace of the decode call that just ran (one kernel launch): the attention
        weights behind every word of the returned caption of each of its `rows` searches, (rows, steps, N), and, unless
        `all_shape` is None, of every beam, all_shape + (steps, N). `valid`: the (rows, S) uint8 mask the caller passed to
        sscvae_select_best_beam, or None."""
        steps, dev = self._max_caption_length, ws.device
        best = torch.empty(rows, steps, num_boxes, dtype=torch.float32, device=dev)
        every = None if all_shape is None else torch.empty(*all_shape, steps, num_boxes, dtype=torch.float32, device=dev)
        stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        _lib.check(_lib.lib().sscvae_decode_attention(self._handle, _lib.ptr(ws), ws.numel(), _lib.ptr(valid), _lib.ptr(every),
                                                      _lib.ptr(best), stream))
        return best, every

    # ------------------------------------------------------------------------------------------
    _STATE_KEYS = ("h1", "c1", "h_encoder", "c_encoder", "h_decoder", "c_decoder")

    def _decode_step(self, image_features, obj_atts, previous_predictions, states, sentiment=None, prior_mean=None,
                     prior_var=None):
        """The reference's eval-mode step function (updown_captioner.py:371-455), which its forward hands to the search as
        `partial(self._decode_step, image_features, obj_atts, sentiment=..., prior_mean=..., prior_var=...)`
        (updown_captioner.py:325-343); `sscvae.ConstrainedBeamSearch` / `BeamSearch` take it the same way.

        previous_predictions: (R,) token ids, R a multiple of B; row r belongs to image r // (R // B). states: the six
        (R, H) tensors of the reference's state dict, or None for zero states. prior_mean / prior_var: (B, Z), or None
        for the prior forward() builds. Returns the reference's eval 5-tuple
        (log_probs (R, V), states, prior_mean (R, Z), prior_log_var (R, Z), attention (R, N)): new fp32 tensors, not
        differentiable; h_encoder / c_encoder pass through (zeros for states=None). One sscvae_decode_step call; the
        per-image state is recomputed only when the features changed (storage, shape, dtype or an in-place edit).

        In training mode with `stepwise_training = True` it is the reference's training step instead: see
        `_train_decode_step`. Without the switch, training mode raises NotImplementedError."""
        if self.training:
            if not self.stepwise_training:
                raise NotImplementedError("_decode_step in training mode needs `stepwise_training = True` (one differentiable "
                                          "step per call); the fused training forward() is the fast training path")
            return self._train_decode_step(image_features, obj_atts, previous_predictions, states, sentiment, prior_mean,
                                           prior_var)
        with torch.no_grad():
            return self._eval_decode_step(image_features, obj_atts, previous_predictions, states, sentiment, prior_mean,
                                          prior_var)

    def _eval_decode_step(self, image_features, obj_atts, previous_predictions, states, sentiment, prior_mean, prior_var):
        self._require_cuda(image_features)
        L = _lib.lib()
        given = image_features
        image_features = self._features(image_features)
        dev = image_features.device
        B, N, F = image_features.shape
        if F != self.image_feature_size:
            raise ValueError(f"image_features last dim {F} != image_feature_size {self.image_feature_size}")
        prev = previous_predictions.to(dev).long().contiguous().view(-1)
        R, H, Z, V = prev.numel(), self.hidden_size, self.z_space, self._vocab_size
        if R == 0 or R % B != 0:
            raise ValueError(f"previous_predictions has {R} rows, not a positive multiple of the batch size {B}")
        # nn.Embedding raises on an out-of-range id; the kernels index the table unchecked (asynchronous: no host sync)
        torch._assert_async(((prev >= 0) & (prev < V)).all(), "previous_predictions contains an id outside [0, vocab_size)")
        if self.sentiment_vae == 1:
            if sentiment is None:
                raise ValueError("sentiment is required when sentiment_vae == 1")
            sentiment = sentiment.to(dev).contiguous().float().view(B, 1)
        else:
            sentiment = None
        obj_means = self._obj_means(obj_atts, B, N, dev)

        def per_image(x, name):
            if x is None:
                return None
            x = x.to(dev).contiguous().float()
            if x.shape != (B, Z):
                raise ValueError(f"{name} must be (B, z_space) = {(B, Z)}, got {tuple(x.shape)}")
            return x
        prior_mean, prior_var = per_image(prior_mean, "prior_mean"), per_image(prior_var, "prior_var")
        if states is None:
            s_in, enc = None, (torch.zeros(R, H, device=dev), torch.zeros(R, H, device=dev))
        else:
            st = {}
            for k in self._STATE_KEYS:
                v = states[k]
                if v.shape != (R, H):
                    raise ValueError(f"states[{k!r}] must be (R, hidden_size) = {(R, H)}, got {tuple(v.shape)}")
                st[k] = v.to(dev).contiguous().float()
            s_in = [st[k] for k in self._STATE_KEYS]
            enc = (states["h_encoder"], states["c_encoder"])
        eps = self._eps_override
        if eps is None and self.rng_mode == "reference":
            eps = torch.randn(R, Z)                                   # one (R,Z) CPU draw per step, like updown_cell.py:206
        if eps is not None:
            eps = eps.to(dev).contiguous().float()
            assert eps.shape == (R, Z)
        nbytes = L.sscvae_decode_step_workspace_bytes(self._handle, B, R, N)
        # one workspace, grown on demand: a search calls with R = B first and R = B*S*K afterwards
        ws = self._ws_cache.get(("step", dev))
        if ws is None or ws.numel() < nbytes:
            ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
            self._ws_cache[("step", dev)] = ws
        # Keyed on the CALLER's tensor: `image_features` is a temporary copy for inputs that are not contiguous fp32 / bf16,
        # and the allocator may hand its block to the next call's copy of different features.
        key = (ws.data_ptr(), given.data_ptr(), given._version, tuple(given.shape), given.dtype, given.stride(),
               self._weights_key(self._weight_tensors()))
        last = getattr(self, "_step_image_state", None)
        reuse = last is not None and last[0] is given and last[1] == key
        self._step_image_state = (given, key)       # keeps the tensor alive: a new one cannot take over its storage
        log_probs = torch.empty(R, V, device=dev)
        h1, c1, hd, cd = (torch.empty(R, H, device=dev) for _ in range(4))
        alpha = torch.empty(R, N, device=dev)
        pm = torch.empty(R, Z, device=dev)
        stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        _lib.check(L.sscvae_set_option(self._handle, b"reuse_image_state", int(reuse)))
        _lib.check(L.sscvae_decode_step(
            self._handle, B, R, N, _lib.ptr(self._packed_weights()), _lib.ptr_array(self._weight_tensors()),
            _lib.ptr(image_features), _lib.ptr(sentiment), _lib.ptr(obj_means), _lib.ptr(prior_mean), _lib.ptr(prior_var),
            _lib.ptr(prev), None if s_in is None else _lib.ptr_array(s_in), _lib.ptr(eps), C.c_uint64(self._next_seed()),
            _lib.ptr(ws), ws.numel(), _lib.ptr(log_probs), _lib.ptr_array([h1, c1, hd, cd]), _lib.ptr(alpha), _lib.ptr(pm),
            stream))
        var = prior_var if prior_var is not None else torch.full((B, Z), float(self.prior_std), device=dev).pow(2)
        prior_log_var = var.log().repeat_interleave(R // B, dim=0)
        new_states = {"h1": h1, "c1": c1, "h_encoder": enc[0], "c_encoder": enc[1], "h_decoder": hd, "c_decoder": cd}
        return log_probs, new_states, pm, prior_log_var, alpha

    def _train_decode_step(self, image_features, obj_atts, previous_predictions, states, sentiment, prior_mean, prior_var):
        """The reference's training-mode step (updown_captioner.py:371-455, updown_cell.py:143-231), one call per timestep of
        its training loop (updown_captioner.py:282-310). One row per image: previous_predictions (B,). states: the six
        (B, H) tensors, or None for zero states; the encoder pair is read. prior_mean / prior_var: (B, Z) or None for the
        prior forward() builds; they only enter the returned prior.

        Returns the reference's training 7-tuple (logits (B,V) raw, states, mean (B,Z), log_var (B,Z), prior_mean (B,Z),
        prior_log_var (B,Z), attention (B,N)), fp32. logits, the states, mean, log_var and attention are differentiable with
        respect to every trainable parameter and the input states, so gradients chain across steps through autograd and
        reach `.grad` by its normal accumulation; with sentiment_vae == 2 the prior mean is differentiable through the
        attention. The prior otherwise passes through in torch (prior_log_var = prior_var.log()), zeros for simple_vae.
        image_features, sentiment and obj_atts get no gradient. Under torch.no_grad(), or when nothing needs a gradient, no
        tape is kept. Each step keeps its own tape, and the per-image state of each feature tensor is a buffer of its
        own, so graphs over different batches can be alive together."""
        self._require_cuda(image_features)
        given = image_features
        image_features = self._features(image_features)
        dev = image_features.device
        B, N, F = image_features.shape
        if F != self.image_feature_size:
            raise ValueError(f"image_features last dim {F} != image_feature_size {self.image_feature_size}")
        prev = previous_predictions.to(dev).long().contiguous().view(-1)
        H, Z, V = self.hidden_size, self.z_space, self._vocab_size
        if prev.numel() != B:
            raise ValueError(f"previous_predictions has {prev.numel()} rows; in training mode it needs one per image ({B})")
        torch._assert_async(((prev >= 0) & (prev < V)).all(), "previous_predictions contains an id outside [0, vocab_size)")
        if self.sentiment_vae == 1:
            if sentiment is None:
                raise ValueError("sentiment is required when sentiment_vae == 1")
            sentiment = sentiment.to(dev).contiguous().float().view(B, 1)
        else:
            sentiment = None
        obj_means = self._obj_means(obj_atts, B, N, dev)
        if states is None:
            st = [None] * 6
        else:
            st = []
            for k in self._STATE_KEYS:
                v = states[k]
                if v.shape != (B, H):
                    raise ValueError(f"states[{k!r}] must be (B, hidden_size) = {(B, H)}, got {tuple(v.shape)}")
                st.append(v.to(dev).contiguous().float())
        eps = self._eps_override
        if eps is None and self.rng_mode == "reference":
            eps = torch.randn(B, Z)                                   # one (B,Z) CPU draw per step, like updown_cell.py:206
        if eps is not None:
            eps = eps.to(dev).contiguous().float()
            assert eps.shape == (B, Z)
        params = self._weight_tensors()
        state = self._train_step_image_state(given, image_features, obj_atts if torch.is_tensor(obj_atts) else obj_means,
                                             obj_means)
        seed = self._next_seed()
        grad = torch.is_grad_enabled() and (any(p.requires_grad for p in params) or
                                            any(t is not None and t.requires_grad for t in st))
        if grad:
            tape = torch.empty(_lib.lib().sscvae_train_step_tape_bytes(self._handle, B, N), dtype=torch.uint8, device=dev)
            outs = _TrainDecodeStep.apply(self, N, state, sentiment, prev, eps, seed, tape, *st, *params)
        else:
            outs = self._train_step_call(N, state, sentiment, prev, None if st[0] is None else st, eps, seed,
                                         self._train_step_workspace(B, N, "tape"))
        logits, s_out, mean, log_var, pm, alpha = outs[0], outs[1:7], outs[7], outs[8], outs[9], outs[10]
        var = prior_var.to(dev).float() if prior_var is not None else torch.full((B, Z), float(self.prior_std), device=dev).pow(2)
        if self.simple_vae:
            pm = torch.zeros(B, Z, device=dev)                                           # updown_cell.py:165-166
        elif self.sentiment_vae != 2:
            if prior_mean is not None:
                pm = prior_mean.to(dev).float()
            elif self.sentiment_vae == 1:
                pm = sentiment.repeat(1, Z) * self.senti_prior_multip                    # updown_captioner.py:250-253
            else:
                pm = torch.zeros(B, Z, device=dev)
        new_states = dict(zip(self._STATE_KEYS, s_out))
        return logits, new_states, mean, log_var, pm, var.log(), alpha

    def _train_step_call(self, N, state, sentiment, prev, states, eps, seed, tape):
        """sscvae_train_step_forward into new output tensors: logits, six states, mean, log_var, prior mean, alpha."""
        B = prev.numel()
        dev = prev.device
        H, Z = self.hidden_size, self.z_space
        logits = torch.empty(B, self._vocab_size, device=dev)
        s_out = [torch.empty(B, H, device=dev) for _ in range(6)]
        mean, log_var = torch.empty(B, Z, device=dev), torch.empty(B, Z, device=dev)
        pm = torch.empty(B, Z, device=dev) if self.sentiment_vae == 2 and not self.simple_vae else torch.empty(0, device=dev)
        alpha = torch.empty(B, N, device=dev)
        ws = self._train_step_workspace(B, N)
        stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        _lib.check(_lib.lib().sscvae_train_step_forward(
            self._handle, B, N, _lib.ptr(self._packed_weights()), _lib.ptr_array(self._weight_tensors()), _lib.ptr(state),
            state.numel(), _lib.ptr(sentiment), _lib.ptr(prev), None if states is None else _lib.ptr_array(states),
            _lib.ptr(eps), C.c_uint64(seed), _lib.ptr(tape), tape.numel(), _lib.ptr(ws), ws.numel(), _lib.ptr(logits),
            _lib.ptr_array(s_out), _lib.ptr(mean), _lib.ptr(log_var), _lib.ptr(pm if pm.numel() else None), _lib.ptr(alpha),
            stream))
        return (logits, *s_out, mean, log_var, pm, alpha)

    def _train_step_workspace(self, B, N, kind="workspace") -> torch.Tensor:
        """The training step's shared scratch (kind "workspace"), or a scratch tape for steps without autograd ("tape")."""
        dev = self._embedding_layer.weight.device
        key = ("step_" + kind, B, N, dev)
        ws = self._ws_cache.get(key)
        if ws is None:
            fn = _lib.lib().sscvae_train_step_workspace_bytes if kind == "workspace" else _lib.lib().sscvae_train_step_tape_bytes
            ws = torch.empty(fn(self._handle, B, N), dtype=torch.uint8, device=dev)
            self._ws_cache = {k: v for k, v in self._ws_cache.items() if k[0] != key[0]}
            self._ws_cache[key] = ws
        return ws

    def _train_step_image_state(self, given, image_features, given_obj, obj_means) -> torch.Tensor:
        """The per-image state of the training step for these features (and obj_means, and the current weights): rebuilt
        into a NEW buffer whenever any of them changed, never in place, because the tapes of earlier steps keep the old
        one. Keyed on the caller's tensors (`given`, `given_obj`), like the eval step's state."""
        B, N, _ = image_features.shape
        ws = self._weight_tensors()
        tkey = lambda t: None if t is None else (t.data_ptr(), t._version, tuple(t.shape), t.dtype, t.stride())
        key = (tkey(given), tkey(given_obj), self._weights_key(ws))
        last = getattr(self, "_train_step_state", None)
        if last is not None and last[0] is given and last[1] is given_obj and last[2] == key:
            return last[3]
        L = _lib.lib()
        dev = image_features.device
        state = torch.empty(L.sscvae_train_step_image_state_bytes(self._handle, B, N), dtype=torch.uint8, device=dev)
        stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        _lib.check(L.sscvae_train_step_image_state(self._handle, B, N, _lib.ptr(self._packed_weights()), _lib.ptr_array(ws),
                                                   _lib.ptr(image_features), _lib.ptr(obj_means), _lib.ptr(state),
                                                   state.numel(), stream))
        self._train_step_state = (given, given_obj, key, state)    # keeps the tensors alive: no new one takes their storage
        return state

    def translate_obj_atts2obj_means(self, obj_atts) -> torch.Tensor:
        """Per-box attribute means of sentiment_vae == 2 (updown_captioner.py:509-532): `obj_atts` holds, per image, one
        `(object, [attribute strings])` entry per box; a box's mean is the average of `mean_choice[first word]` over its
        attributes that have an entry (zeros when none has), boxes are zero-padded to the longest image and the result is
        scaled by `latent_embedding_multip`. Returns (B, max boxes, Z) fp32 on the CPU."""
        if self.mean_choice is None:
            raise ValueError("sentiment_vae == 2 with attribute lists needs `mean_choice` ({word: (Z,) vector})")
        Z = self.z_space
        per_image = []
        for boxes in obj_atts:
            rows = torch.zeros(len(boxes), Z, dtype=torch.float64)
            for i, box in enumerate(boxes):
                hits = [self.mean_choice[a.split(" ")[0]] for a in box[1] if a.split(" ")[0] in self.mean_choice]
                if hits:
                    rows[i] = torch.stack([torch.as_tensor(h, dtype=torch.float64).reshape(-1) for h in hits]).mean(dim=0)
            per_image.append(rows)
        out = torch.zeros(len(per_image), max(len(r) for r in per_image), Z, dtype=torch.float64)
        for i, rows in enumerate(per_image):
            out[i, :len(rows)] = rows
        return (out * self.latent_embedding_multip).float()

    def _obj_means(self, obj_atts, B, N, device):
        """(B, N, Z) fp32 device tensor for sentiment_vae == 2 (a tensor is taken as already translated), else None."""
        if self.sentiment_vae != 2 or self.simple_vae:
            return None
        if obj_atts is None:
            raise ValueError("obj_atts is required when sentiment_vae == 2")
        if not torch.is_tensor(obj_atts):
            obj_atts = self.translate_obj_atts2obj_means(obj_atts)
        obj_atts = obj_atts.to(device).contiguous().float()
        if obj_atts.shape != (B, N, self.z_space):
            # the reference multiplies (B, N) attention weights with it (updown_cell.py:161-163): one row per box
            raise ValueError(f"obj_atts must be (B, num_boxes, z_space) = {(B, N, self.z_space)}, got {tuple(obj_atts.shape)}")
        return obj_atts

    @torch.no_grad()
    def sample(self, image_features: torch.Tensor, sentiment=None, n_samples: int = 100, obj_atts=None, fsm=None,
               num_constraints=None, constraints=None, constraint2states=None):
        """Diverse sampling: `n_samples` captions per image with independent latent draws, in one call.

        Replaces the reference's inference loop `for k in range(N_Z_SAMPLES): model(image_features, ...)`
        (var_updown/scripts/inference.py:138-167) over the eval branch: same per-sample computation
        (`_decode_step` with z ~ N(prior_mean, prior_var), updown_cell.py:200-208), but the n_samples sequences of an
        image share its region features and run as rows of one batch.

        use_cbs=False: beam-1 search. Returns {"predictions": (B, n_samples, steps) int64, "log_probs": (B, n_samples)};
        `fsm` must be None.

        use_cbs=True: one constrained beam search (beam_size, per_node_beam_size) per (image, sample), exactly what
        n_samples calls of forward() on single images would run; see `_sample_search`. Returns
        {"predictions": (B, n_samples, n) int64, "n_steps": (B, n_samples) int64}.

        return_attention: both results gain "attention", (B, n_samples, n, N) fp32, the attention weights over the boxes
        behind every word (zero after the caption's first boundary token)."""
        self._require_cuda(image_features)
        if self._use_cbs:
            return self._sample_search(image_features, sentiment, n_samples, obj_atts, fsm, num_constraints, constraints,
                                       constraint2states)
        if fsm is not None:
            raise ValueError("fsm is only used with use_cbs=True; sample() without it is the unconstrained beam-1 path")
        L = _lib.lib()
        image_features = self._features(image_features)
        dev = image_features.device
        B, N, F = image_features.shape
        if F != self.image_feature_size:
            raise ValueError(f"image_features last dim {F} != image_feature_size {self.image_feature_size}")
        J, steps = int(n_samples), self._max_caption_length
        if J < 1:
            raise ValueError("n_samples must be >= 1")
        if self.sentiment_vae == 1:
            if sentiment is None:
                raise ValueError("sentiment is required when sentiment_vae == 1")
            sentiment = sentiment.to(dev).contiguous().float().view(B, 1)
        else:
            sentiment = None
        obj_means = self._obj_means(obj_atts, B, N, dev)
        eps = self._eps_override
        if eps is not None:
            eps = eps.to(dev).contiguous().float()
            assert eps.shape == (steps, B * J, self.z_space)
        nbytes = L.sscvae_decode_samples_workspace_bytes(self._handle, B, J, N)
        key = ("decode", B, N, -J, 1, dev)
        ws = self._ws_cache.get(key)
        if ws is None:
            self._ws_cache = {k: v for k, v in self._ws_cache.items() if k[0] != "decode"}
            ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
            self._ws_cache[key] = ws
        okey = ("decode_out", B, -J, 1, steps, dev)                # persistent outputs: stable pointers for graph replay
        outs = self._ws_cache.get(okey)
        if outs is None:
            outs = (torch.empty(B, J, steps, dtype=torch.long, device=dev), torch.empty(B, J, dtype=torch.float32, device=dev),
                    torch.zeros(1, dtype=torch.int32, device=dev))
            self._ws_cache[okey] = outs
        preds, scores, n_steps = outs
        stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        self._reuse_image_state(key, image_features)
        _lib.check(L.sscvae_decode_samples(
            self._handle, B, J, N, _lib.ptr(self._packed_weights()), _lib.ptr_array(self._weight_tensors()),
            _lib.ptr(image_features), _lib.ptr(sentiment), _lib.ptr(obj_means), _lib.ptr(eps), C.c_uint64(self._next_seed()),
            _lib.ptr(ws), nbytes, _lib.ptr(preds), _lib.ptr(scores), _lib.ptr(n_steps), stream))
        att = self._decode_attention(ws, None, N, B * J)[0] if self.return_attention else None
        n = int(n_steps.item())
        out = {"predictions": preds[..., :n].clone(), "log_probs": scores.clone()}
        if att is not None:
            out["attention"] = att.view(B, J, steps, N)[:, :, :n].contiguous()
        return out

    def _sample_search(self, image_features, sentiment, n_samples, obj_atts, fsm, num_constraints, constraints,
                       constraint2states):
        """sample() with use_cbs=True: the reference's loop `for k in range(N_Z_SAMPLES): model(image_features, ...,
        fsm=..., num_constraints=...)` (inference.py:138-167) in one call (sscvae_decode_samples_search).

        Every (image b, sample j) is one constrained beam search with its own latent draws, and it stops when its own
        beams have all emitted the boundary token, as the reference's batch-1 call does (cbs.py:167).
        - `fsm`: the reference's (B,S,S,V) uint8 tensor or an `FsmBits` (B,S,V) table, shared by the samples of an image;
          or (B*n_samples, ...), row b*n_samples + j being sample j's own machine. `num_constraints` has as many rows.
        - cbs_simple=False: `constraints` / `constraint2states` hold one entry per FSM row (valid_states_with_attributes).
        - `_eps_override`: (steps, B*n_samples*S*K, Z) normals, step 0 reading row (b*n_samples + j)*S*K. Otherwise the
          device Philox stream; rng_mode "reference" does not apply here (as in the beam-1 sample()).
        - Workspace: the fp32 logits of all R = B*n_samples*S*K rows are materialised, R*V*4 bytes (16 images x 20
          samples x S 8 x K 5 at V 10 000: 512 MB); sscvae_decode_samples_search_workspace_bytes gives the total.
        Returns {"predictions": (B, n_samples, n), "n_steps": (B, n_samples)} int64 with n = the largest n_steps; a
        sample's entries after its own n_steps are the boundary token. `last_search` holds every beam:
        {"predictions": (B,J,S,K,n), "log_probs": (B,J,S,K), "n_steps": (B,J)}, plus "attention" (B,J,S,K,n,N) with
        return_attention."""
        from .fsm import FsmBits, valid_states_with_attributes
        L = _lib.lib()
        image_features = self._features(image_features)
        dev = image_features.device
        B, N, F = image_features.shape
        if F != self.image_feature_size:
            raise ValueError(f"image_features last dim {F} != image_feature_size {self.image_feature_size}")
        J, K, P, steps, V = int(n_samples), self.beam_size, self.per_node_beam_size, self._max_caption_length, self._vocab_size
        if J < 1:
            raise ValueError("n_samples must be >= 1")
        if self.sentiment_vae == 1:
            if sentiment is None:
                raise ValueError("sentiment is required when sentiment_vae == 1")
            sentiment = sentiment.to(dev).contiguous().float().view(B, 1)
        else:
            sentiment = None
        obj_means = self._obj_means(obj_atts, B, N, dev)
        if fsm is None:
            raise ValueError("fsm is required when use_cbs=True")
        fsm_packed = isinstance(fsm, FsmBits)
        if fsm_packed:                                               # bit table built on the device (fsm.build_fsm_bits)
            fsm = fsm.bits
            T, S = fsm.shape[0], fsm.shape[1]
            if fsm.shape != (T, S, V) or T not in (B, B * J) or fsm.device != dev or not fsm.is_contiguous():
                raise ValueError(f"FsmBits must be a contiguous (B or B*n_samples, S, V) table on {dev}, got {tuple(fsm.shape)}")
        else:
            fsm = fsm.to(dev).to(torch.uint8).contiguous()
            T, S = fsm.shape[0], fsm.shape[1]
            if fsm.dim() != 4 or fsm.shape != (T, S, S, V) or T not in (B, B * J):
                raise ValueError(f"fsm must be (B or B*n_samples, S, S, V), got {tuple(fsm.shape)}")
        per_sample = int(T != B)
        if num_constraints is None:
            nc = torch.zeros(T, dtype=torch.long, device=dev)
        else:
            nc = num_constraints.to(dev).long().contiguous().view(-1)
            if nc.numel() != T:
                raise ValueError(f"num_constraints must have one entry per FSM ({T}), got {nc.numel()}")
        valid = None
        if not self.cbs_simple:
            # object / attribute rule (decoding.py:87-123), per machine, then per search
            if constraints is None or constraint2states is None:
                raise ValueError("cbs_simple=False needs `constraints` and `constraint2states`")
            counts = [int(n) for n in nc.cpu()]
            mask = torch.zeros(T, S, dtype=torch.uint8)
            for i in range(T):
                states = valid_states_with_attributes(counts[i], constraints[i], constraint2states[i],
                                                      self._min_constraints_to_satisfy)
                if not states:
                    raise ValueError(f"FSM {i}: no state satisfies the constraints")
                mask[i, states] = 1
            valid = (mask if per_sample else mask.repeat_interleave(J, dim=0)).contiguous().to(dev)
        R = B * J * S * K
        eps = self._eps_override
        if eps is not None:
            eps = eps.to(dev).contiguous().float()
            assert eps.shape == (steps, R, self.z_space)
        nbytes = L.sscvae_decode_samples_search_workspace_bytes(self._handle, B, J, N, S, K, per_sample)
        if nbytes == 0:
            raise ValueError(f"unsupported search shape: states {S}, beam {K} (1..32 states, beam 1..8)")
        key = ("decode", B, N, S, K, dev, J, per_sample)
        ws = self._ws_cache.get(key)
        if ws is None:
            self._ws_cache = {k: v for k, v in self._ws_cache.items() if k[0] != "decode"}
            ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
            self._ws_cache[key] = ws
        okey = ("decode_out", B, S, K, steps, dev, J)               # persistent outputs: stable pointers for graph replay
        outs = self._ws_cache.get(okey)
        if outs is None:
            outs = (torch.empty(B, J, S, K, steps, dtype=torch.long, device=dev),
                    torch.empty(B, J, S, K, dtype=torch.float32, device=dev),
                    torch.empty(B, J, steps, dtype=torch.long, device=dev), torch.zeros(B, J, dtype=torch.int32, device=dev))
            self._ws_cache[okey] = outs
        preds, scores, best, n_steps = outs
        stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        self._reuse_image_state(key, image_features)
        _lib.check(L.sscvae_set_option(self._handle, b"fsm_packed", int(fsm_packed)))
        _lib.check(L.sscvae_decode_samples_search(
            self._handle, B, J, N, S, K, P, _lib.ptr(self._packed_weights()), _lib.ptr_array(self._weight_tensors()),
            _lib.ptr(image_features), _lib.ptr(sentiment), _lib.ptr(obj_means), _lib.ptr(fsm), per_sample, _lib.ptr(nc),
            int(self._min_constraints_to_satisfy), _lib.ptr(eps), C.c_uint64(self._next_seed()), _lib.ptr(ws), nbytes,
            _lib.ptr(preds), _lib.ptr(scores), _lib.ptr(best), _lib.ptr(n_steps), stream))
        if valid is not None:
            _lib.check(L.sscvae_select_best_beam(_lib.ptr(preds), _lib.ptr(scores), _lib.ptr(valid), B * J, S, K, steps,
                                                 _lib.ptr(best), stream))
        if self.return_attention:
            att, every = self._decode_attention(ws, valid, N, B * J, (B, J, S, K))
        ns = n_steps.long()
        n = int(ns.max().item())                                    # each search's own early exit (cbs.py:167)
        self.last_search = {"predictions": preds[..., :n].clone(), "log_probs": scores.clone(), "n_steps": ns.clone()}
        out = {"predictions": best[..., :n].clone(), "n_steps": ns.clone()}
        if self.return_attention:
            self.last_search["attention"] = every[..., :n, :].contiguous()
            out["attention"] = att.view(B, J, steps, N)[:, :, :n].contiguous()
        return out

    def sample_search_region(self, B, N, J, S, K, fsm_per_sample, name, dtype, shape):
        """Typed view of a named region of the last sample() workspace with use_cbs=True (tests / debugging)."""
        off, nb = C.c_size_t(), C.c_size_t()
        _lib.check(_lib.lib().sscvae_decode_samples_search_region(self._handle, B, J, N, S, K, int(fsm_per_sample),
                                                                  name.encode(), C.byref(off), C.byref(nb)))
        ws = self._ws_cache[("decode", B, N, S, K, self._embedding_layer.weight.device, J, int(fsm_per_sample))]
        n = 1
        for s in shape:
            n *= s
        itemsize = torch.empty(0, dtype=dtype).element_size()
        assert n * itemsize <= nb.value, (name, n * itemsize, nb.value)
        return ws[off.value: off.value + n * itemsize].view(dtype).view(*shape)

    @torch.no_grad()
    def _decode(self, image_features, sentiment, fsm, num_constraints, obj_means=None, constraints=None,
                constraint2states=None):
        L = _lib.lib()
        dev = image_features.device
        B, N, _ = image_features.shape
        K, P, steps = self.beam_size, self.per_node_beam_size, self._max_caption_length
        if self._use_cbs:
            if fsm is None:
                raise ValueError("fsm is required when use_cbs=True")
            from .fsm import FsmBits, valid_states_with_attributes
            fsm_packed = isinstance(fsm, FsmBits)
            if fsm_packed:                                           # bit table built on the device (fsm.build_fsm_bits)
                fsm = fsm.bits
                S = fsm.shape[1]
                if fsm.shape != (B, S, self._vocab_size) or fsm.device != dev or not fsm.is_contiguous():
                    raise ValueError(f"FsmBits must be a contiguous (B,S,V) table on {dev}, got {tuple(fsm.shape)}")
            else:
                fsm = fsm.to(dev).to(torch.uint8).contiguous()
                S = fsm.shape[1]
                if fsm.shape != (B, S, S, self._vocab_size):
                    raise ValueError(f"fsm must be (B,S,S,V), got {tuple(fsm.shape)}")
            nc = None if num_constraints is None else num_constraints.to(dev).long().contiguous()
            if nc is None:
                nc = torch.zeros(B, dtype=torch.long, device=dev)
            valid = None
            if not self.cbs_simple:
                # object / attribute rule (decoding.py:87-123): the valid end states come from host-side bookkeeping
                if constraints is None or constraint2states is None:
                    raise ValueError("cbs_simple=False needs `constraints` and `constraint2states`")
                counts = [int(n) for n in (num_constraints if num_constraints is not None else [0] * B)]
                mask = torch.zeros(B, S, dtype=torch.uint8)
                for i in range(B):
                    states = valid_states_with_attributes(counts[i], constraints[i], constraint2states[i],
                                                          self._min_constraints_to_satisfy)
                    if not states:
                        raise ValueError(f"image {i}: no state satisfies the constraints")
                    mask[i, states] = 1
                valid = mask.to(dev)
        else:
            S, fsm, nc, valid, fsm_packed = 1, None, None, None, False
        R = B * S * K
        eps = self._eps_override
        if eps is None and self.rng_mode == "reference":
            e = torch.zeros(steps, R, self.z_space)
            e[0, ::S * K] = torch.randn(B, self.z_space)            # first step: one row per image (cbs.py:127)
            for t in range(1, steps):
                e[t] = torch.randn(R, self.z_space)
            eps = e
        if eps is not None:
            eps = eps.to(dev).contiguous().float()
            assert eps.shape == (steps, R, self.z_space)
        nbytes = L.sscvae_decode_workspace_bytes(self._handle, B, N, S, K)
        key = ("decode", B, N, S, K, dev)
        ws = self._ws_cache.get(key)
        if ws is None:
            self._ws_cache = {k: v for k, v in self._ws_cache.items() if k[0] != "decode"}
            ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
            self._ws_cache[key] = ws
        okey = ("decode_out", B, S, K, steps, dev)                 # persistent outputs: stable pointers for graph replay
        outs = self._ws_cache.get(okey)
        if outs is None:
            outs = (torch.empty(B, S, K, steps, dtype=torch.long, device=dev), torch.empty(B, S, K, dtype=torch.float32, device=dev),
                    torch.empty(B, steps, dtype=torch.long, device=dev), torch.zeros(1, dtype=torch.int32, device=dev))
            self._ws_cache[okey] = outs
        preds, scores, best, n_steps = outs
        stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        self._reuse_image_state(key, image_features)
        _lib.check(L.sscvae_set_option(self._handle, b"fsm_packed", int(fsm_packed)))
        _lib.check(L.sscvae_decode(
            self._handle, B, N, S, K, P, _lib.ptr(self._packed_weights()), _lib.ptr_array(self._weight_tensors()),
            _lib.ptr(image_features), _lib.ptr(sentiment), _lib.ptr(obj_means), _lib.ptr(fsm), _lib.ptr(nc),
            int(self._min_constraints_to_satisfy), _lib.ptr(eps), C.c_uint64(self._next_seed()), _lib.ptr(ws), nbytes,
            _lib.ptr(preds), _lib.ptr(scores), _lib.ptr(best), _lib.ptr(n_steps), stream))
        if valid is not None:
            _lib.check(L.sscvae_select_best_beam(_lib.ptr(preds), _lib.ptr(scores), _lib.ptr(valid), B, S, K, steps,
                                                 _lib.ptr(best), stream))
        attention = None
        if self.return_attention:
            attention, every = self._decode_attention(ws, valid, N, B, (B, S, K))
        n = int(n_steps.item())                                     # the reference's data-dependent early exit (cbs.py:167)
        self.last_search = {"predictions": preds[..., :n].clone(), "log_probs": scores.clone(), "n_steps": n}
        if attention is not None:
            self.last_search["attention"] = every[..., :n, :].contiguous()
            attention = attention[:, :n].contiguous()
        return best[:, :n].clone(), attention
