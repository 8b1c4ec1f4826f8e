"""Drop-in ``ModelBiLSTM`` whose forward runs in libdsp_b200 (sm_100a CUDA kernels).

Mirrors ``deepsignal_plant/models.py:99-240`` of the reference: same constructor
(``:103-106``), same ``forward(kmer, base_means, base_stds, base_signal_lens, signals) ->
(logits, probs)`` (``:178-240``), same ``state_dict`` keys (the parameters live in
same-named ``nn.Embedding`` / ``nn.LSTM`` / ``nn.Linear`` containers created in the same
order, so ``torch.manual_seed`` + construction reproduces the reference's initial weights
and ``load_state_dict`` / ``model_dict.update(para_dict)`` work unchanged,
``call_modifications.py:219-223``), ``init_hidden`` (``:169-176``), ``get_model_type``.

Differences, all deliberate:

* Training is opt-in: ``ModelBiLSTM(..., trainable=True)`` in ``train()`` mode runs ``forward`` through
  the fp32 training kernels (``csrc/kernels_train.cu``) inside a ``torch.autograd.Function``, so the
  reference's loop (``train.py:104-128``) works as written.  Without ``trainable=True``, ``forward`` in
  ``train()`` mode raises as before.  ``eval()`` always runs the inference path of ``precision``.
* Inputs must be CUDA tensors on the module's device -- there is no CPU path.
* Initial LSTM states.  The reference draws fresh ``torch.randn`` states on every call
  (``models.py:169-176``).  ``state_mode`` selects how this module gets them:
  ``"philox"`` (default) draws N(0,1) on the device (Philox4x32-10) -- statistically the
  same, no host RNG, no 16 KB/site PCIe traffic; ``"init_hidden"`` calls
  ``self.init_hidden`` three times in the reference's order (seq, signal, comb), which
  consumes the torch CPU generator exactly like the reference and is what the parity
  tests use.  Overriding ``init_hidden`` on an instance or subclass selects the second
  mode automatically.
"""
from __future__ import annotations

import ctypes as C
import os

import torch
import torch.nn as nn

from . import _native


class ModelBiLSTM(nn.Module):
    def __init__(self, seq_len=13, signal_len=16, num_layers1=3, num_layers2=1, num_classes=2,
                 dropout_rate=0.5, hidden_size=256,
                 vocab_size=16, embedding_size=4, is_base=True, is_signallen=True,
                 module="both_bilstm", device=0, precision=None, max_batch=65536,
                 state_mode="philox", seed=0, trainable=False):
        super().__init__()
        self.model_type = "BiLSTM"
        self.module = module
        self.device = device
        self.seq_len = seq_len
        self.signal_len = signal_len
        self.num_layers1 = num_layers1
        self.num_layers2 = num_layers2
        self.num_classes = num_classes
        self.hidden_size = hidden_size
        self.vocab_size = vocab_size
        self.embedding_size = embedding_size

        if module == "both_bilstm":
            self.nhid_seq = hidden_size // 2
            self.nhid_signal = hidden_size - self.nhid_seq
        elif module == "seq_bilstm":
            self.nhid_seq = hidden_size
        elif module == "signal_bilstm":
            self.nhid_signal = hidden_size
        else:
            raise ValueError("--model_type is not right!")

        # parameter containers: created in the reference's order (models.py:131-161)
        if module != "signal_bilstm":
            self.embed = nn.Embedding(vocab_size, embedding_size)
            self.is_base = is_base
            self.is_signallen = is_signallen
            self.sigfea_num = 3 if is_signallen else 2
            in_seq = (embedding_size if is_base else 0) + self.sigfea_num
            self.lstm_seq = nn.LSTM(in_seq, self.nhid_seq, num_layers2, dropout=dropout_rate,
                                    batch_first=True, bidirectional=True)
            self.fc_seq = nn.Linear(self.nhid_seq * 2, self.nhid_seq)
        else:
            self.is_base = is_base
            self.is_signallen = is_signallen
        if module != "seq_bilstm":
            self.lstm_signal = nn.LSTM(signal_len, self.nhid_signal, num_layers2, dropout=dropout_rate,
                                       batch_first=True, bidirectional=True)
            self.fc_signal = nn.Linear(self.nhid_signal * 2, self.nhid_signal)
        self.lstm_comb = nn.LSTM(hidden_size, hidden_size, num_layers1, dropout=dropout_rate,
                                 batch_first=True, bidirectional=True)
        self.fc1 = nn.Linear(hidden_size * 2, hidden_size)
        self.fc2 = nn.Linear(hidden_size, num_classes)

        precision = precision or os.environ.get("DSP_B200_PRECISION", "auto")
        if precision == "auto":
            # the tcgen05 kernels cover the shapes the reference ships models for (hidden 256);
            # anything else runs on the fp32 CUDA-core kernels
            kseq = (embedding_size if is_base else 0) + (3 if is_signallen else 2)
            precision = "fp16" if (hidden_size == 256 and signal_len <= 64 and kseq <= 16) else "fp32"
        self.precision = precision
        if self.precision not in _native.PRECISIONS:
            raise ValueError("precision must be one of %s" % sorted(_native.PRECISIONS))
        self.max_batch = int(max_batch)
        self.state_mode = state_mode
        self.seed = int(seed)
        self.dropout_rate = float(dropout_rate)
        self.trainable = bool(trainable)
        self.last_dropout_masks = None
        self._calls = 0
        self._handle = None
        self._handle_device = None
        self._packed_key = None
        self.last_labels = None

    # ---- reference API ----------------------------------------------------------------
    def get_model_type(self):
        return self.model_type

    def init_hidden(self, batch_size, num_layers, hidden_size):
        """``models.py:169-176``: N(0,1) states from the torch CPU generator, moved to the
        module's device."""
        dev = self._param_device()
        h0 = torch.randn(num_layers * 2, batch_size, hidden_size)
        c0 = torch.randn(num_layers * 2, batch_size, hidden_size)
        if dev.type == "cuda":
            h0 = h0.cuda(dev)
            c0 = c0.cuda(dev)
        return h0, c0

    # ---- native handle ----------------------------------------------------------------
    def _apply(self, fn, *args, **kwargs):
        # .cuda() / .to() / .float(): parameters may be swapped for new objects -- forget the cached list
        self.__dict__.pop("_plist", None)
        return super()._apply(fn, *args, **kwargs)

    def _param_device(self):
        return next(self.parameters()).device

    def _uses_init_hidden(self):
        return (self.state_mode == "init_hidden" or "init_hidden" in self.__dict__
                or type(self).init_hidden is not ModelBiLSTM.init_hidden)

    def _destroy(self):
        if getattr(self, "_handle", None):
            try:
                _native.lib().dsp_destroy(self._handle)
            except Exception:
                pass
            self._handle = None
            self._packed_key = None

    def __del__(self):
        self._destroy()

    def _create_handle(self, dev):
        L = _native.lib()
        if self._handle is not None and self._handle_device != dev.index:
            self._destroy()
        if self._handle is None:
            cfg = _native.DspConfig(
                seq_len=self.seq_len, signal_len=self.signal_len, num_layers1=self.num_layers1,
                num_layers2=self.num_layers2, num_classes=self.num_classes, hidden_size=self.hidden_size,
                vocab_size=self.vocab_size, embedding_size=self.embedding_size,
                is_base=int(bool(self.is_base)), is_signallen=int(bool(self.is_signallen)),
                module=_native.MODULES[self.module], device=dev.index,
                precision=_native.PRECISIONS[self.precision], reserved=0, max_batch=self.max_batch)
            h = C.c_void_p()
            _native.check(L.dsp_create(C.byref(h), C.byref(cfg)), "dsp_create")
            self._handle = h
            self._handle_device = dev.index
            self._packed_key = None
        return self._handle

    def _ensure_handle(self, dev):
        self._create_handle(dev)
        # the Parameter objects persist across .cuda() / load_state_dict (their data pointer / version change): keep the
        # list instead of walking the module tree on every forward
        plist = self.__dict__.get("_plist")
        if plist is None:
            plist = self.__dict__["_plist"] = list(self.parameters())
        key = tuple((p.data_ptr(), p._version) for p in plist)
        if key != self._packed_key:
            self.pack_weights()
            self._packed_key = key
        return self._handle

    def pack_weights(self):
        """Hand the current state_dict to the library and convert it to the kernel layouts
        (runs automatically when parameters change; cheap enough to call explicitly)."""
        L = _native.lib()
        for name, t in self.state_dict().items():
            a = t.detach().to("cpu", torch.float32).contiguous()
            _native.check(L.dsp_set_param(self._handle, name.encode(), a.data_ptr(), a.numel()),
                          "dsp_set_param(%s)" % name)
        _native.check(L.dsp_pack_weights(self._handle), "dsp_pack_weights")

    # ---- forward ----------------------------------------------------------------------
    def _prep(self, t, dev, shape):
        if t is None:
            return None
        if not torch.is_tensor(t):
            raise TypeError("ModelBiLSTM.forward expects torch tensors")
        if t.device != dev:
            raise RuntimeError("input tensor is on %s but the model is on %s; there is no CPU path"
                               % (t.device, dev))
        return t.detach().reshape(shape).to(torch.float32).contiguous()

    def _init_hidden_states(self, n, dev):
        """``init_hidden`` for the seq, signal and comb stacks in the reference's order -> (6 device
        pointers for the library, the tensors behind them)."""
        has_seq = self.module != "signal_bilstm"
        has_sig = self.module != "seq_bilstm"
        keep = []
        ptrs = (C.c_void_p * 6)()
        groups = ((has_seq, self.num_layers2, getattr(self, "nhid_seq", 0)),
                  (has_sig, self.num_layers2, getattr(self, "nhid_signal", 0)),
                  (True, self.num_layers1, self.hidden_size))
        for g, (used, layers, hid) in enumerate(groups):
            if not used:
                continue
            h0, c0 = self.init_hidden(n, layers, hid)
            h0 = h0.detach().to(dev, torch.float32).contiguous()
            c0 = c0.detach().to(dev, torch.float32).contiguous()
            if tuple(h0.shape) != (layers * 2, n, hid) or tuple(c0.shape) != (layers * 2, n, hid):
                raise RuntimeError("init_hidden returned shape %s, expected %s"
                                   % (tuple(h0.shape), (layers * 2, n, hid)))
            keep += [h0, c0]
            ptrs[2 * g], ptrs[2 * g + 1] = h0.data_ptr(), c0.data_ptr()
        return ptrs, keep

    def dropout_mask_shapes(self, n):
        """Shapes of the dropout-mask slots of ``dsp_train_forward`` for n sites, ``None`` for a slot this
        module never uses: nn.LSTM inter-layer dropout of lstm_seq, lstm_signal, lstm_comb (every layer's
        output but the last), then the head's dropout before and after fc1 (models.py:234-237)."""
        T, H = self.seq_len, self.hidden_size
        has_seq = self.module != "signal_bilstm"
        has_sig = self.module != "seq_bilstm"
        shapes = [(n, T, 2 * self.nhid_seq) if has_seq else None] * (self.num_layers2 - 1)
        shapes += [(n, T, 2 * self.nhid_signal) if has_sig else None] * (self.num_layers2 - 1)
        shapes += [(n, T, 2 * H)] * (self.num_layers1 - 1)
        return shapes + [(n, 2 * H), (n, H)]

    def draw_dropout_masks(self, n, dev):
        """keep / (1 - p) masks drawn with torch's CUDA generator (``torch.rand >= p``), as nn.Dropout
        scales them; all ``None`` when ``dropout_rate`` is 0."""
        p = self.dropout_rate
        if p <= 0:
            return [None] * len(self.dropout_mask_shapes(n))
        return [None if shp is None else (torch.rand(shp, device=dev) >= p).to(torch.float32).div_(1.0 - p)
                for shp in self.dropout_mask_shapes(n)]

    def forward(self, kmer, base_means, base_stds, base_signal_lens, signals):
        if self.training and self.trainable:
            return self._forward_train(kmer, base_means, base_stds, base_signal_lens, signals)
        if self.training:
            raise RuntimeError("deepsignal_plant_b200.ModelBiLSTM implements inference only; "
                               "call .eval() (training is outside the accelerated hot path)")
        dev = self._param_device()
        if dev.type != "cuda":
            raise RuntimeError("ModelBiLSTM parameters are on %s; move the model to a CUDA device "
                               "(.cuda(device)) -- this implementation has no CPU fallback" % dev)
        T, S = self.seq_len, self.signal_len
        has_seq = self.module != "signal_bilstm"
        has_sig = self.module != "seq_bilstm"
        kmer = self._prep(kmer, dev, (-1, T)) if has_seq else None
        means = self._prep(base_means, dev, (-1, T)) if has_seq else None
        stds = self._prep(base_stds, dev, (-1, T)) if has_seq else None
        lens = self._prep(base_signal_lens, dev, (-1, T)) if has_seq else None
        sig = self._prep(signals, dev, (-1, T, S)) if has_sig else None
        n = (kmer if has_seq else sig).shape[0]
        with torch.cuda.device(dev):
            handle = self._ensure_handle(dev)
            states_arg, keep = self._init_hidden_states(n, dev) if self._uses_init_hidden() else (None, [])
            logits = torch.empty((n, self.num_classes), dtype=torch.float32, device=dev)
            probs = torch.empty((n, self.num_classes), dtype=torch.float32, device=dev)
            labels = torch.empty((n,), dtype=torch.int32, device=dev)
            stream = torch.cuda.current_stream(dev).cuda_stream
            self._calls += 1
            ptr = lambda t: None if t is None else t.data_ptr()
            _native.check(_native.lib().dsp_forward(
                handle, ptr(kmer), ptr(means), ptr(stds), ptr(lens), ptr(sig), states_arg,
                (self.seed << 20) + self._calls, n, logits.data_ptr(), probs.data_ptr(),
                labels.data_ptr(), stream), "dsp_forward")
            # tensors handed to the asynchronous call must outlive it on this stream
            for t in keep + [x for x in (kmer, means, stds, lens, sig) if x is not None]:
                t.record_stream(torch.cuda.current_stream(dev))
        self.last_labels = labels
        return logits, probs

    def _forward_train(self, kmer, base_means, base_stds, base_signal_lens, signals):
        dev = self._param_device()
        if dev.type != "cuda":
            raise RuntimeError("ModelBiLSTM parameters are on %s; move the model to a CUDA device "
                               "(.cuda(device)) -- this implementation has no CPU fallback" % dev)
        T, S = self.seq_len, self.signal_len
        has_seq = self.module != "signal_bilstm"
        has_sig = self.module != "seq_bilstm"
        inputs = (self._prep(kmer, dev, (-1, T)) if has_seq else None,
                  self._prep(base_means, dev, (-1, T)) if has_seq else None,
                  self._prep(base_stds, dev, (-1, T)) if has_seq else None,
                  self._prep(base_signal_lens, dev, (-1, T)) if has_seq else None,
                  self._prep(signals, dev, (-1, T, S)) if has_sig else None)
        n = (inputs[0] if has_seq else inputs[4]).shape[0]
        with torch.cuda.device(dev):
            handle = self._create_handle(dev)
            states_arg, keep = self._init_hidden_states(n, dev) if self._uses_init_hidden() else (None, [])
            masks = self.draw_dropout_masks(n, dev)
            self.last_dropout_masks = masks
            self._calls += 1
            params = [p for p in self.state_dict(keep_vars=True).values()]
            for p in params:
                if p.dtype != torch.float32 or not p.is_contiguous():
                    raise RuntimeError("training needs contiguous float32 parameters")
            logits = _TrainStep.apply(handle, inputs, states_arg, keep, masks, (self.seed << 20) + self._calls, *params)
        return logits, torch.softmax(logits, 1)

    # ---- host-buffer entry (the FloatTensor/.cpu() boundary of _call_mods) ---------------
    def forward_host(self, kmer, base_means, base_stds, base_signal_lens, signals):
        """numpy float32 arrays in host memory -> (logits, probs, labels) numpy arrays.
        Stages through pinned buffers with H2D/D2H overlapped with compute
        (``dsp_forward_host``); initial states are Philox-drawn on the device."""
        import numpy as np
        dev = self._param_device()
        if dev.type != "cuda":
            raise RuntimeError("ModelBiLSTM parameters are on %s; this implementation has no CPU fallback" % dev)
        if self.training:
            raise RuntimeError("inference only; call .eval()")
        T, S = self.seq_len, self.signal_len
        has_seq = self.module != "signal_bilstm"
        has_sig = self.module != "seq_bilstm"

        def prep(a, shape):
            return np.ascontiguousarray(np.asarray(a, dtype=np.float32).reshape(shape))
        k = prep(kmer, (-1, T)) if has_seq else None
        m = prep(base_means, (-1, T)) if has_seq else None
        s = prep(base_stds, (-1, T)) if has_seq else None
        ln = prep(base_signal_lens, (-1, T)) if has_seq else None
        sg = prep(signals, (-1, T, S)) if has_sig else None
        n = (k if has_seq else sg).shape[0]
        logits = np.empty((n, self.num_classes), np.float32)
        probs = np.empty((n, self.num_classes), np.float32)
        labels = np.empty((n,), np.int32)
        ptr = lambda a: None if a is None else a.ctypes.data
        with torch.cuda.device(dev):
            handle = self._ensure_handle(dev)
            self._calls += 1
            _native.check(_native.lib().dsp_forward_host(
                handle, ptr(k), ptr(m), ptr(s), ptr(ln), ptr(sg), (self.seed << 20) + self._calls, n,
                logits.ctypes.data, probs.ctypes.data, labels.ctypes.data), "dsp_forward_host")
        return logits, probs, labels

    # ---- streaming form of forward_host: page-locked buffers, submissions overlap ------------
    def submit_host(self, kmer, base_means, base_stds, base_signal_lens, signals, logits, probs, labels=None):
        """Enqueue one batch held in PAGE-LOCKED host memory (``torch`` tensors created with
        ``pin_memory()``/``pin_memory=True``, float32 contiguous; ``labels`` int32) and return a
        ticket immediately; ``logits``/``probs``/``labels`` (pinned outputs the caller owns) are
        valid after ``wait_host(ticket)``.  Submissions run in order, and batch i+1's host->device
        copies overlap batch i's kernels (``dsp_forward_host_submit``)."""
        dev = self._param_device()
        if dev.type != "cuda":
            raise RuntimeError("ModelBiLSTM parameters are on %s; this implementation has no CPU fallback" % dev)
        if self.training:
            raise RuntimeError("inference only; call .eval()")
        has_seq = self.module != "signal_bilstm"
        has_sig = self.module != "seq_bilstm"

        def chk(t, dtype):
            if t is None:
                return None
            if not (torch.is_tensor(t) and t.device.type == "cpu" and t.is_pinned() and t.is_contiguous() and t.dtype == dtype):
                raise ValueError("submit_host needs contiguous page-locked CPU tensors of dtype %s" % dtype)
            return t.data_ptr()
        n = (kmer if has_seq else signals).shape[0]
        args = [chk(x, torch.float32) if used else None for x, used in
                ((kmer, has_seq), (base_means, has_seq), (base_stds, has_seq), (base_signal_lens, has_seq), (signals, has_sig))]
        if tuple(logits.shape) != (n, self.num_classes) or tuple(probs.shape) != (n, self.num_classes):
            raise ValueError("output tensors must be (n, num_classes)")
        outs = [chk(logits, torch.float32), chk(probs, torch.float32), chk(labels, torch.int32)]
        ticket = C.c_int64(-1)
        with torch.cuda.device(dev):
            handle = self._ensure_handle(dev)
            self._calls += 1
            _native.check(_native.lib().dsp_forward_host_submit(
                handle, *args, (self.seed << 20) + self._calls, n, *outs, C.byref(ticket)), "dsp_forward_host_submit")
        return int(ticket.value)

    def wait_host(self, ticket):
        _native.check(_native.lib().dsp_forward_host_wait(self._handle, int(ticket)), "dsp_forward_host_wait")

    def launch_count(self):
        return int(_native.lib().dsp_launch_count(self._handle)) if self._handle else 0


def _ptr_array(tensors):
    arr = (C.c_void_p * max(1, len(tensors)))()
    for i, t in enumerate(tensors):
        arr[i] = None if t is None else t.data_ptr()
    return arr


class _TrainStep(torch.autograd.Function):
    """logits = ModelBiLSTM forward in train() mode on the fp32 training kernels; backward hands dlogits to
    ``dsp_train_backward``.  The activation arena is a torch tensor kept in the context, so several forwards
    may precede one backward and the memory returns to torch's allocator with the graph."""

    @staticmethod
    def forward(ctx, handle, inputs, states_arg, keep, masks, seed, *params):
        L = _native.lib()
        n = (inputs[0] if inputs[0] is not None else inputs[4]).shape[0]
        dev = params[0].device
        C_ = params[-1].shape[0]
        arena = torch.empty(int(L.dsp_train_arena_bytes(handle, n)), dtype=torch.uint8, device=dev)
        logits = torch.empty((n, C_), dtype=torch.float32, device=dev)
        pp, mp = _ptr_array(params), _ptr_array(masks)
        ptr = lambda t: None if t is None else t.data_ptr()
        stream = torch.cuda.current_stream(dev).cuda_stream
        _native.check(L.dsp_train_forward(handle, pp, len(params), *(ptr(t) for t in inputs), states_arg, seed, mp, n,
                                          arena.data_ptr(), logits.data_ptr(), stream), "dsp_train_forward")
        ctx.handle, ctx.n, ctx.arena, ctx.masks = handle, n, arena, masks
        ctx.save_for_backward(*params)
        return logits

    @staticmethod
    def backward(ctx, dlogits):
        L = _native.lib()
        params = ctx.saved_tensors
        dev = params[0].device
        dlogits = dlogits.to(torch.float32).contiguous()
        ws = torch.empty(int(L.dsp_train_workspace_bytes(ctx.handle, ctx.n)), dtype=torch.uint8, device=dev)
        grads = [torch.empty_like(p) for p in params]
        stream = torch.cuda.current_stream(dev).cuda_stream
        _native.check(L.dsp_train_backward(ctx.handle, _ptr_array(params), len(params), _ptr_array(ctx.masks),
                                           ctx.arena.data_ptr(), dlogits.data_ptr(), ctx.n, ws.data_ptr(),
                                           _ptr_array(grads), stream), "dsp_train_backward")
        return (None,) * 6 + tuple(grads)
