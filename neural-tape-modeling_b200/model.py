"""Drop-in replacements for the three hot-path classes of the reference's code/model.py:

    RNN                    code/model.py:20-246    (forward / predict / warm_start / hidden handling)
    TimeVaryingDelayLine   code/model.py:249-332
    DiffDelRNN             code/model.py:335-653

Same constructor arguments, attribute names, state_dict keys and method signatures, so
`from model import RNN, DiffDelRNN, TimeVaryingDelayLine` in code/test-model.py:29 can point here.
All arithmetic runs in libntm_b200.so (hand-written sm_100a CUDA) behind the C ABI of include/ntm_b200.h, reached
through the PyTorch C++ extension ntm_b200_torch.so (torch.ops.ntm.*, csrc/torch_binding.cpp: CUDAGuard on the
input's device, PyTorch's current stream, TORCH_CHECK on a non-zero return code); torch only owns the memory and the
stream.  The host-buffer pipeline (predict_host) and the resident real-time server bind the same C ABI with ctypes.
There is no CPU path and no torch.nn.GRU fallback: tensors must live on a CUDA device, otherwise a RuntimeError is
raised.  Training (train_epoch / validate, code/model.py:90-216, :426-616) is out of scope.

Deliberate differences from the reference (SURVEY.md section 8b):
  * the device is the input tensor's device, not the global "cuda" (needed to shard streams over 8 GPUs);
  * predict() accepts B > 1 streams: the batch-1 warm state (and silence-response delay history) is broadcast,
    which equals B separate reference predict() calls; it runs ONE persistent launch instead of 2048-sample
    segments (the recurrence is segmentation-invariant);
  * forward() rejects C != 1 channels (the reference's reshape is only a transpose when C == 1).
"""
import ctypes
import weakref

import torch

from . import lib as _lib

WARM_LEN = 2 ** 10      # code/model.py:60, :386
ENGINE_H = 64           # state width of the kernels (ntm::H64); smaller hidden sizes run zero-padded


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _stream(device):
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _host_out(out, shape, name, dtype=torch.float32):
    """Result buffer of a *_host call: a fresh pinned tensor, or the caller's contiguous host tensor of that dtype."""
    if out is None:
        return torch.empty(shape, dtype=dtype, pin_memory=True)
    if out.is_cuda or out.dtype != dtype or tuple(out.shape) != tuple(shape) or not out.is_contiguous():
        raise RuntimeError(f"{name}: expected a contiguous {dtype} host tensor of shape {tuple(shape)}")
    return out


def _as_rows(t, name):
    """(B, 1, T) tensor -> float32 view with unit stride in T; returns (tensor, B, T, ld)."""
    if t.dim() != 3 or t.shape[1] != 1:
        raise RuntimeError(f"{name}: expected shape (N_BATCHES, 1, N_SAMPLES), got {tuple(t.shape)}")
    if not t.is_cuda:
        raise RuntimeError(f"{name}: ntm_b200 has no CPU path; move the tensor to a CUDA device")
    if t.dtype != torch.float32:
        t = t.float()                                   # code/model.py:76, :403 (f64 -> f32)
    if t.shape[2] > 1 and t.stride(2) != 1:
        t = t.contiguous()
    B, T = t.shape[0], t.shape[2]
    ld = t.stride(0) if B > 1 else max(T, 1)
    if B > 1 and ld < T:
        t = t.contiguous()
        ld = T
    return t, B, T, ld


class _Engine:
    """Owns the packed-parameter handle of one module on one device; re-prepared when parameters change.

    Change detection: data_ptr + the autograd version counter of every parameter.  Inference tensors (modules built or
    moved under torch.inference_mode()) carry no version counter: for them an in-place edit of a parameter is not seen --
    call `module.refresh_parameters()` after one (load_state_dict / .to() / .float() always re-pack)."""

    def __init__(self):
        self.handle = None          # int (a Handle* of the C ABI)
        self.generation = 0         # bumped whenever the handle is released: live BlockStreams re-resolve theirs
        self._params = ()
        self._ptrs = ()
        self._versions = None       # None: inference tensors, no version counters
        self._device = None
        self._finalizer = None

    def _stale(self, params, device):
        if self.handle is None or device != self._device:
            return True
        for p, q, ptr in zip(params, self._params, self._ptrs):
            if p is not q or (p is not None and p.data_ptr() != ptr):
                return True
        if self._versions is not None:
            for p, v in zip(params, self._versions):
                if p is not None and p._version != v:
                    return True
        return False

    def get(self, gru, head, device):
        params = (gru.weight_ih_l0, gru.weight_hh_l0, gru.bias_ih_l0, gru.bias_hh_l0, head.weight, head.bias)
        if self._stale(params, device):
            self.release()
            H = params[1].shape[1]
            if params[0].shape[1] != 1 or head.weight.shape[0] != 1:
                raise RuntimeError("ntm_b200: only input_size=1, output_size=1 models are supported")
            if not 1 <= H <= ENGINE_H:
                raise RuntimeError(f"ntm_b200: the engine is built for hidden_size <= {ENGINE_H} (all shipped checkpoints are "
                                   f"GRU-HS[64]; smaller models run zero-padded to 64 units, exactly); this module has "
                                   f"hidden_size={H}")
            ops = _lib.ops()
            handle = int(ops.prepare(*[p.detach() if p is not None else None for p in params], device.index))
            self.handle, self._device = handle, device
            self._params, self._ptrs = params, tuple(None if p is None else p.data_ptr() for p in params)
            try:
                self._versions = tuple(None if p is None else p._version for p in params)
            except RuntimeError:            # inference tensors carry no version counter
                self._versions = None
            self._finalizer = weakref.finalize(self, ops.destroy, handle)
        return self.handle

    def __deepcopy__(self, memo):          # handles are per-object; a copied module re-prepares lazily
        return _Engine()

    def __reduce__(self):
        return (_Engine, ())

    def release(self):
        if self._finalizer is not None:
            self._finalizer()               # drops this module's reference (an open real-time stream keeps its own)
            self._finalizer = None
        self.handle, self._params, self._ptrs = None, (), ()
        self.generation += 1


class RNN(torch.nn.Module):
    """GRU(1 -> hidden) + Linear(hidden -> 1) tape nonlinearity; mirrors code/model.py:20-246."""

    _head_bias = True

    def __init__(self, input_size=1, hidden_size=8, output_size=1, skip=False):
        super().__init__()
        self.input_size = input_size
        self.hidden_size = hidden_size
        self.output_size = output_size
        self.skip = skip
        # parameter containers only (state_dict keys GRU.* / output.*); their forward() is never called
        self.GRU = torch.nn.GRU(input_size, hidden_size, batch_first=True)
        self.output = torch.nn.Linear(hidden_size, output_size, bias=self._head_bias)
        # "fp32" exact CUDA-core | "f16x3" (alias "strict") fp32-grade on tensor cores | "f16" | "tf32" | "bf16" rounded
        # operands (include/ntm_b200.h NTM_MODE_*)
        self.mode = "fp32"
        # True: forward() writes into per-shape buffers it keeps (the returned tensor is overwritten by the next call of
        # the same shape) -- no allocation per call, and the call sequence can be captured in a CUDA Graph
        self.static_io = False
        self._io = {}
        self._engine = _Engine()
        self.hidden = None
        # parameters are re-packed lazily whenever they may have changed
        self.register_load_state_dict_post_hook(lambda module, incompatible: module._engine.release())

    def _apply(self, fn, *args, **kwargs):      # .to() / .cuda() / .float() ...
        self._engine.release()
        self._io = {}
        return super()._apply(fn, *args, **kwargs)

    def refresh_parameters(self):
        """Re-pack the parameters at the next call (needed only after an in-place edit of an inference-mode parameter)."""
        self._engine.release()

    # -- state handling (code/model.py:50-56) ---------------------------------------------------
    def initialize_hidden(self):
        self.hidden = None

    def detach_hidden(self):
        self.hidden = self.hidden.clone().detach()

    def _device(self):
        return self.GRU.weight_hh_l0.device

    def _handle(self, device):
        if self._device() != device:
            raise RuntimeError(f"input is on {device} but the model parameters are on {self._device()}")
        return self._engine.get(self.GRU, self.output, device)

    def _hidden_in(self, B, device):
        """self.hidden checked like torch.nn.GRU checks it, as the engine's (1, B, 64) state (see _to_engine)."""
        h = self.hidden
        if h is None:
            return None
        if tuple(h.shape) != (1, B, self.hidden_size):
            raise RuntimeError(f"Expected hidden size (1, {B}, {self.hidden_size}), got {list(h.shape)}")
        if h.device != device or h.dtype != torch.float32 or not h.is_contiguous():
            h = h.to(device, torch.float32).contiguous()
        return self._to_engine(h)

    # The engine's state is always ENGINE_H = 64 units wide.  A model with hidden_size < 64 runs zero-padded: the padded units
    # have zero weights in and out, so their state stays 0 (r = z = 1/2, n = tanh(0) = 0) and no real unit ever sees them --
    # the result is the hidden_size-wide GRU's, term for term.  `self.hidden` keeps the reference's (1, B, hidden_size) shape.
    def _to_engine(self, h):
        if h is None or h.shape[-1] == ENGINE_H:
            return h
        return torch.nn.functional.pad(h, (0, ENGINE_H - h.shape[-1]))

    def _from_engine(self, h):
        if h is None or self.hidden_size == ENGINE_H:
            return h
        return h[..., :self.hidden_size].contiguous()

    def warm_start(self):
        """1024 samples of silence from the current state, batch 1 (code/model.py:58-65)."""
        with torch.no_grad():
            self(torch.zeros((1, 1, WARM_LEN), device=self._device()))

    def forward(self, x):
        """x (N_BATCHES, 1, N_SAMPLES) -> y of the same shape; carries self.hidden (code/model.py:67-88)."""
        if not (x.dtype is torch.float32 and x.is_cuda and x.dim() == 3 and x.shape[1] == 1 and x.stride(2) == 1):
            x = _as_rows(x, "x")[0]
        dev = x.device
        handle = self._handle(dev)
        B = x.shape[0]
        h_in = self.hidden
        if h_in is not None and not (h_in.shape[1] == B and h_in.shape[2] == ENGINE_H and h_in.device == dev
                                     and h_in.dtype is torch.float32 and h_in.is_contiguous()):
            h_in = self._hidden_in(B, dev)
        ops = _lib.ops()
        if self.static_io:
            key = (B, x.shape[2], dev)
            buf = self._io.get(key)
            if buf is None:
                buf = self._io[key] = (torch.empty((B, 1, x.shape[2]), dtype=torch.float32, device=dev),
                                       torch.empty((1, B, ENGINE_H), dtype=torch.float32, device=dev))
            y, h_out = buf
            ops.gru_forward_out(handle, _lib.MODES[self.mode], x, h_in, y, h_out, bool(self.skip))
        else:
            y, h_out = ops.gru_forward(handle, _lib.MODES[self.mode], x, h_in, bool(self.skip))
        self.hidden = h_out if self.hidden_size == ENGINE_H else self._from_engine(h_out)
        return y

    def block_stream(self, n_streams=1, block_len=64):
        """Real-time block mode (BASELINE.json cfg 5): consecutive `forward` calls on short blocks with carried state,
        with the per-call host work stripped to one C call -- see BlockStream."""
        return BlockStream(self, n_streams, block_len)

    def realtime_stream(self, n_streams=1, block_len=64, idle_timeout_ms=5000):
        """Real-time block mode with a resident kernel (host blocks in, host blocks out) -- see RealtimeStream."""
        return RealtimeStream(self, n_streams, block_len, idle_timeout_ms)

    def predict(self, input):
        """Zero state -> warm start -> whole signal (code/model.py:218-246), for any number of streams."""
        dev = self._device()
        input = input.to(dev)
        self.initialize_hidden()
        self.warm_start()
        B = input.shape[0]
        if B != 1:
            self.hidden = self.hidden.expand(1, B, self.hidden_size).contiguous()
        return self.forward(input)

    def predict_host(self, input, chunk=0, out=None):
        """predict() for a HOST tensor (pinned for full speed): chunked H2D / kernel / D2H pipeline inside the
        engine (ntm_gru_predict_host).  Returns a pinned host tensor (`out` if given: page-locking a fresh
        multi-GB result buffer costs seconds, so repeated callers pass their own).  This is the end-to-end call the
        bench times (host->device at code/test-model.py:427-433, device->host at :525).

        A float16 `input` selects the opt-in 16-bit host transport (ntm_gru_predict_host_f16): the samples cross the
        host link as binary16 -- half the bytes -- and the result comes back as float16; arithmetic and state stay as
        `mode` says."""
        if input.is_cuda or input.dim() != 3 or input.shape[1] != 1:
            raise RuntimeError("predict_host expects a host tensor of shape (N_BATCHES, 1, N_SAMPLES)")
        dev = self._device()
        handle = self._handle(dev)
        half = input.dtype == torch.float16
        x = input.contiguous() if half else input.float().contiguous()
        B, T = x.shape[0], x.shape[2]
        self.initialize_hidden()
        self.warm_start()
        h = self._to_engine(self.hidden).reshape(1, ENGINE_H).expand(B, ENGINE_H).contiguous().cpu()
        y = _host_out(out, (B, 1, T), "out", torch.float16 if half else torch.float32)
        fn = _lib.load().ntm_gru_predict_host_f16 if half else _lib.load().ntm_gru_predict_host
        rc = fn(handle, _lib.MODES[self.mode], _ptr(x), _ptr(y), _ptr(h), B, T, int(bool(self.skip)), int(chunk))
        _lib.check(rc)
        self.hidden = self._from_engine(h.reshape(1, B, ENGINE_H)).to(dev)
        return y


class BlockStream:
    """Block-by-block processing of `n_streams` streams with the state carried on the device.

    Semantically identical to calling `model(x_block)` repeatedly (code/model.py:67-88 with `self.hidden` carried,
    SURVEY.md section 9.3 #1): the state starts from `model.hidden` (zeros if None, i.e. after `initialize_hidden()`;
    call `warm_start()` first for `predict()` semantics) and is written back by `close()`.  Buffers, raw pointers, the
    handle and the CUDA stream are resolved once, so a block costs one ctypes call + one kernel launch."""

    def __init__(self, model, n_streams, block_len):
        dev = model._device()
        if dev.type != "cuda":
            raise RuntimeError("ntm_b200 has no CPU path; move the model to a CUDA device")
        self.model, self.B, self.T, self.device = model, int(n_streams), int(block_len), dev
        self._dev = dev.index
        self._resolve_handle()
        self._mode = _lib.MODES[model.mode]
        self._skip = int(bool(model.skip))
        h = model._hidden_in(self.B, dev)
        self.h = torch.zeros((1, self.B, ENGINE_H), dtype=torch.float32, device=dev) if h is None else h.clone()
        self.y = torch.empty((self.B, 1, self.T), dtype=torch.float32, device=dev)
        self._ld_out = max(self.T, 1)                       # row stride of the internal output buffers
        self._fn = _lib.load().ntm_gru_forward
        self._hp = ctypes.c_void_p(self.h.data_ptr())
        self._yp = ctypes.c_void_p(self.y.data_ptr())
        self._st = _stream(dev)

    def _resolve_handle(self):
        """The model's packed-parameter handle; called again once the parameters were re-packed (load_state_dict, .to(),
        ...), which frees the old one."""
        self._handle = ctypes.c_void_p(self.model._handle(self.device))
        self._generation = self.model._engine.generation

    def _ld(self, t, name, min_len=0):
        """Row stride of `t`, a float32 block of shape (n_streams, 1, min_len .. block_len) on the model's device with unit
        stride in time."""
        if t.dtype != torch.float32 or t.get_device() != self._dev or t.dim() != 3 or t.shape[0] != self.B \
                or t.shape[1] != 1 or not min_len <= t.shape[2] <= self.T or t.stride(2) != 1:
            raise RuntimeError(f"{name}: expected a float32 CUDA block of shape ({self.B}, 1, {min_len} .. {self.T}) on "
                               f"{self.device}")
        return t.stride(0) if self.B > 1 else max(t.shape[2], 1)

    def process(self, x, out=None):
        """x (n_streams, 1, block_len) float32 on the model's device -> y (the internal buffer, overwritten by the
        next call, or `out`, at least as long as x).  Asynchronous on the stream that was current when the BlockStream
        was created."""
        ldx = self._ld(x, "x")
        T = x.shape[2]
        if out is None:
            y, yp, ldy = self.y, self._yp, self._ld_out
        else:
            y, yp, ldy = out, ctypes.c_void_p(out.data_ptr()), self._ld(out, "out", T)
        if self._generation != self.model._engine.generation:
            self._resolve_handle()
        rc = self._fn(self._handle, self._mode, ctypes.c_void_p(x.data_ptr()), ldx, yp, ldy, self._hp, self._hp, self.B, T,
                      self._skip, self._st)
        if rc:
            _lib.check(rc)
        return y if T == y.shape[2] else y[:, :, :T]

    def close(self):
        """Hand the carried state back to the model (`model.hidden`)."""
        self.model.hidden = self.model._from_engine(self.h)
        return self.model.hidden


class RealtimeStream:
    """Block-by-block processing of up to 4 streams through a RESIDENT server kernel (ntm_rt_*, csrc/gru_mma.cu RT form).

    Same semantics as BlockStream / repeated `model(x_block)` calls with carried `self.hidden` (code/model.py:67-88), but
    blocks live in HOST memory (a real-time audio callback): `process(x)` takes a float32 host tensor or numpy array of
    shape (n_streams, block_len) [or (n_streams, 1, block_len)] and returns the output block as a host tensor of the same
    shape.  A block costs two PCIe round trips plus the kernel's own steps -- no launch, no prologue, no stream
    synchronisation.  The state starts from `model.hidden` and is handed back by `close()`.  Tensor-core modes only.
    While the stream is open do not synchronise the whole device (torch.cuda.synchronize()): the resident kernel only
    ends at `close()` or after `idle_timeout_ms` without a block."""

    def __init__(self, model, n_streams=1, block_len=64, idle_timeout_ms=5000):
        dev = model._device()
        if dev.type != "cuda":
            raise RuntimeError("ntm_b200 has no CPU path; move the model to a CUDA device")
        self.model, self.B, self.T, self.device = model, int(n_streams), int(block_len), dev
        h = model._hidden_in(self.B, dev)
        h_host = None if h is None else h.reshape(self.B, ENGINE_H).to("cpu", torch.float32).contiguous()
        torch.cuda.current_stream(dev).synchronize()         # the state above is final before the server reads its copy
        self._rt = ctypes.c_void_p()
        _lib.check(self._open(h_host, int(idle_timeout_ms)))
        self._y = torch.empty((self.B, self.T), dtype=torch.float32)
        self._fn = _lib.load().ntm_rt_process
        self._yp = ctypes.c_void_p(self._y.data_ptr())
        self.x_in = torch.zeros((self.B, self.T), dtype=torch.float32)       # optional fixed input block for step()
        self._xp = ctypes.c_void_p(self.x_in.data_ptr())

    def _open(self, h_host, idle_timeout_ms):
        m = self.model
        return _lib.load().ntm_rt_open(m._handle(self.device), _lib.MODES[m.mode], _ptr(h_host), self.B, self.T,
                                       int(bool(m.skip)), idle_timeout_ms, ctypes.byref(self._rt))

    def _live(self):
        """The open server's stream pointer."""
        if self._rt is None:
            raise RuntimeError("ntm_b200: real-time stream is closed")
        return self._rt

    def _host_block(self, b, name):
        t = torch.as_tensor(b)
        if t.is_cuda or t.dtype != torch.float32 or t.numel() != self.B * self.T or not t.is_contiguous():
            raise RuntimeError(f"{name}: expected contiguous float32 HOST blocks of {self.B} x {self.T} samples")
        return t

    def step(self):
        """Lowest-overhead form: process the block the caller wrote into `self.x_in`; returns the internal output
        block (overwritten by the next call)."""
        rc = self._fn(self._live(), self._xp, self._yp)
        if rc:
            _lib.check(rc)
        return self._y

    def process(self, x):
        rt = self._live()
        xt = self._host_block(x, "x")
        rc = self._fn(rt, ctypes.c_void_p(xt.data_ptr()), self._yp)
        if rc:
            _lib.check(rc)
        return self._y.reshape(xt.shape)

    def _stop(self, h=None):
        """Stop the resident kernel; the final state goes into the host tensor `h` (None: dropped)."""
        rt, self._rt = self._rt, None
        _lib.check(_lib.load().ntm_rt_close(rt, _ptr(h)))

    def close(self):
        """Stop the resident kernel and hand the carried state back to the model (`model.hidden`)."""
        if self._rt is not None:
            h = torch.empty((self.B, ENGINE_H), dtype=torch.float32)
            self._stop(h)
            self.model.hidden = self.model._from_engine(h.reshape(1, self.B, ENGINE_H)).to(self.device)
        return self.model.hidden

    def __del__(self):
        try:
            if getattr(self, "_rt", None) is not None:
                self._stop()
        except Exception:
            pass


class TimeVaryingDelayLine(torch.nn.Module):
    """Feed-forward linear-interpolation delay line with carried history; mirrors code/model.py:249-332."""

    def __init__(self, max_delay=40000, channels=1):
        super().__init__()
        self.max_delay = max_delay
        self.check_delay = True     # keep the reference's assert (costs one stream sync per call)
        # plain attribute, not a registered buffer: stays out of state_dict (code/model.py:267)
        self.buffer = torch.zeros(2, channels, max_delay)

    def _history(self, B, device):
        buf = self.buffer
        if buf.dim() != 3 or buf.shape[0] != B or buf.shape[1] != 1:
            raise RuntimeError(f"Sizes of tensors must match: delay buffer {list(buf.shape)} vs batch {B}")
        if buf.shape[2] != self.max_delay:
            raise RuntimeError(f"delay buffer length {buf.shape[2]} != max_delay {self.max_delay}")
        if buf.device != device or buf.dtype != torch.float32 or not buf.is_contiguous():
            buf = buf.to(device, torch.float32).contiguous()
        return buf

    def _check(self, d):
        """The reference's `assert self.max_delay >= torch.max(dt)` (code/model.py:283); NaN trips it too."""
        if self.check_delay and d.shape[2] > 0:
            if d.is_cuda:
                ok = _lib.ops().delay_check(d, int(self.max_delay))
            else:
                ok = bool((d <= float(self.max_delay)).all())
            if not ok:
                raise AssertionError("delay exceeds max_delay (history length)")

    def forward(self, x, dt, warmup=False):
        """x, dt (N_BATCHES, 1, N_SAMPLES), dt in samples -> delayed x (code/model.py:269-320)."""
        x, B, T, ldx = _as_rows(x, "x")
        dt, Bd, Td, ldd = _as_rows(dt.to(x.device), "dt")
        if (Bd, Td) != (B, T):
            raise RuntimeError(f"x {tuple(x.shape)} and dt {tuple(dt.shape)} must have the same shape")
        hist = self._history(B, x.device)
        self._check(dt)
        y, self.buffer = _lib.ops().delay_forward(x, dt, hist, bool(warmup))
        return y

    def detach_buffer(self):
        self.buffer = self.buffer.clone().detach()

    def init_buffer(self, N, max_d=None):
        """Zero history for N streams (code/model.py:326-332).  max_d defaults to the current max_delay so that
        apply_delay's one-argument call (code/test-model.py:268) works."""
        if max_d is not None:
            self.max_delay = max_d
        device = torch.device("cuda") if torch.cuda.is_available() else torch.device("cpu")
        self.buffer = torch.zeros(N, 1, self.max_delay, device=device)


class DiffDelRNN(RNN):
    """GRU + bias-free Linear head + time-varying delay line; mirrors code/model.py:335-653."""

    _head_bias = False

    def __init__(self, input_size=1, hidden_size=8, output_size=1, skip=False, max_delay=10000):
        super().__init__(input_size, hidden_size, output_size, skip)
        self.max_delay = max_delay
        self.diffdel = TimeVaryingDelayLine(max_delay=max_delay)
        self.initialize_hidden(2, max_delay)

    def initialize_hidden(self, N=2, max_D=None):
        """Zero state and a zero delay history of length int(max_D)+1 (code/model.py:372-375)."""
        self.hidden = None
        if hasattr(self, "diffdel"):
            self.diffdel.init_buffer(N, int(self.max_delay if max_D is None else max_D) + 1)

    def detach_hidden(self):
        super().detach_hidden()
        self.diffdel.detach_buffer()

    def warm_start(self):
        """GRU + delay line on 1024 samples of silence with zero delay, batch 1 (code/model.py:377-391)."""
        with torch.no_grad():
            z = torch.zeros((1, 1, WARM_LEN), device=self._device())
            self(z, z.clone())

    def forward(self, x, del_traj, warmup=False):
        """-> (y, pre_d): GRU head output before and after the delay (code/model.py:393-424)."""
        x, B, T, ldx = _as_rows(x, "x")
        dev = x.device
        d, Bd, Td, ldd = _as_rows(del_traj.to(dev), "del_traj")
        if (Bd, Td) != (B, T):
            raise RuntimeError(f"x {tuple(x.shape)} and del_traj {tuple(d.shape)} must have the same shape")
        handle = self._handle(dev)
        h_in = self._hidden_in(B, dev)
        hist = self.diffdel._history(B, dev)
        self.diffdel._check(d)
        y, pre_d, h_out, self.diffdel.buffer = _lib.ops().diffdel_forward(
            handle, _lib.MODES[self.mode], x, d, h_in, hist, bool(warmup), bool(self.skip))
        self.hidden = self._from_engine(h_out)
        return y, pre_d

    def predict(self, input, d_traj):
        """-> (output, output_pre_d) (code/model.py:618-653), for any number of streams."""
        dev = self._device()
        input, d_traj = input.to(dev), d_traj.to(dev)
        B = input.shape[0]
        self.initialize_hidden(1, self.max_delay)
        self.warm_start()
        if B != 1:
            self.hidden = self.hidden.expand(1, B, self.hidden_size).contiguous()
            self.diffdel.buffer = self.diffdel.buffer.expand(B, 1, -1).contiguous()
        return self.forward(input, d_traj)

    def predict_host(self, input, d_traj, chunk=0, out=None, out_pre_d=None):
        """predict() for HOST tensors through ntm_diffdel_predict_host; returns pinned host (output, output_pre_d)
        (`out` / `out_pre_d` if given)."""
        if input.is_cuda or d_traj.is_cuda or input.dim() != 3 or input.shape[1] != 1:
            raise RuntimeError("predict_host expects host tensors of shape (N_BATCHES, 1, N_SAMPLES)")
        dev = self._device()
        handle = self._handle(dev)
        x = input.float().contiguous()
        d = d_traj.float().contiguous()
        B, T = x.shape[0], x.shape[2]
        self.diffdel._check(d)                      # the assert forward() makes (code/model.py:283), on the host copy
        self.initialize_hidden(1, self.max_delay)
        self.warm_start()
        D = int(self.diffdel.max_delay)
        h = self._to_engine(self.hidden).reshape(1, ENGINE_H).expand(B, ENGINE_H).contiguous().cpu()
        hist = self.diffdel.buffer.reshape(1, D).expand(B, D).contiguous().cpu()
        y = _host_out(out, (B, 1, T), "out")
        pre = _host_out(out_pre_d, (B, 1, T), "out_pre_d")
        rc = _lib.load().ntm_diffdel_predict_host(handle, _lib.MODES[self.mode], _ptr(x), _ptr(d), _ptr(y), _ptr(pre),
                                                  _ptr(h), _ptr(hist), B, T, D, int(bool(self.skip)), int(chunk))
        _lib.check(rc)
        self.hidden = self._from_engine(h.reshape(1, B, ENGINE_H)).to(dev)
        self.diffdel.buffer = hist.reshape(B, 1, D).to(dev)
        return y, pre

    def block_stream(self, n_streams=1, block_len=64):
        """Real-time block mode of the full tape model: consecutive `forward(x, d)` calls on short blocks with state and
        delay history carried on the device, one C call per block -- see DelayBlockStream."""
        return DelayBlockStream(self, n_streams, block_len)

    def realtime_stream(self, n_streams=1, block_len=64, idle_timeout_ms=5000):
        """Real-time block mode of the full tape model with a resident kernel (host blocks in, host blocks out) -- see
        RealtimeDelayStream."""
        return RealtimeDelayStream(self, n_streams, block_len, idle_timeout_ms)


class DelayBlockStream(BlockStream):
    """Block-by-block DiffDelRNN processing of `n_streams` streams with the state and the delay history carried on the
    device.

    Semantically identical to calling `model(x_block, d_block)` repeatedly (code/model.py:393-424 with `self.hidden` and
    `self.diffdel.buffer` carried): both start from the model (`initialize_hidden(B, max_D)`, `warm_start()` and a
    broadcast to B streams first give `predict()` semantics) and are written back by `close()`.  Buffers, raw pointers, the
    handle and the CUDA stream are resolved once, so a block costs one ctypes call and one engine launch while the last
    D + 129 samples of pre_d fit on chip (DESIGN.md 3.6; three launches otherwise: GRU, delay read, history roll); the history
    alternates between two device buffers because hist_out must not alias hist_in.  When
    `model.diffdel.check_delay` is set (the default), every block first runs the reference's delay assert, which
    synchronises the stream once per block; a refused block raises AssertionError and changes nothing."""

    def __init__(self, model, n_streams, block_len):
        super().__init__(model, n_streams, block_len)
        self.D = int(model.diffdel.max_delay)
        hist = model.diffdel._history(self.B, self.device)
        self.hist = (hist.clone(), torch.empty_like(hist))
        self._cur = 0                                       # self.hist[_cur] holds the carried history
        self.pre_d = torch.empty_like(self.y)
        L = _lib.load()
        self._fn, self._check = L.ntm_diffdel_forward, L.ntm_delay_check
        self._pp = ctypes.c_void_p(self.pre_d.data_ptr())
        self._histp = tuple(ctypes.c_void_p(t.data_ptr()) for t in self.hist)

    def process(self, x, d, out=None, out_pre_d=None):
        """x, d (n_streams, 1, block_len) float32 on the model's device -> (y, pre_d): the internal buffers, overwritten
        by the next call, or `out` / `out_pre_d`, at least as long as x.  Asynchronous on the stream that was current when
        the stream was created, except for the delay check."""
        ldx, ldd = self._ld(x, "x"), self._ld(d, "d")
        if d.shape != x.shape:
            raise RuntimeError(f"x {tuple(x.shape)} and d {tuple(d.shape)} must have the same shape")
        T = x.shape[2]
        if out is None:
            y, yp, ldy = self.y, self._yp, self._ld_out
        else:
            y, yp, ldy = out, ctypes.c_void_p(out.data_ptr()), self._ld(out, "out", T)
        if out_pre_d is None:
            pre, pp, ldp = self.pre_d, self._pp, self._ld_out
        else:
            pre, pp, ldp = out_pre_d, ctypes.c_void_p(out_pre_d.data_ptr()), self._ld(out_pre_d, "out_pre_d", T)
        if self._generation != self.model._engine.generation:
            self._resolve_handle()
        dp = ctypes.c_void_p(d.data_ptr())
        if self.model.diffdel.check_delay and T > 0:
            rc = self._check(dp, ldd, self.B, T, self.D, self._dev, self._st)
            if rc:
                _lib.check(rc)
        rc = self._fn(self._handle, self._mode, ctypes.c_void_p(x.data_ptr()), ldx, dp, ldd, yp, ldy, pp, ldp, self._hp,
                      self._hp, self._histp[self._cur], self._histp[self._cur ^ 1], self.B, T, self.D, 0, self._skip,
                      self._st)
        if rc:
            _lib.check(rc)
        self._cur ^= 1
        if T != y.shape[2]:
            y, pre = y[:, :, :T], pre[:, :, :T]
        return y, pre

    def close(self):
        """Hand the carried state and delay history back to the model (`model.hidden`, `model.diffdel.buffer`)."""
        self.model.diffdel.buffer = self.hist[self._cur]
        return super().close(), self.model.diffdel.buffer


class RealtimeDelayStream(RealtimeStream):
    """Block-by-block DiffDelRNN processing of up to 4 streams through a RESIDENT server kernel (ntm_rt_diffdel_*,
    csrc/gru_mma.cu RT + delay form).

    Same semantics as DelayBlockStream / repeated `model(x_block, d_block)` calls with `self.hidden` and
    `self.diffdel.buffer` carried (code/model.py:393-424), with the blocks in HOST memory like RealtimeStream: the GRU,
    the head and the wow/flutter delay line run in one persistent CTA that keeps the last samples of pre_d on chip across
    blocks.  `process(x, d)` takes float32 host tensors or numpy arrays of shape (n_streams, block_len) [or (n_streams, 1,
    block_len)] and returns host (y, pre_d) of the same shape.  State and history start from the model and are handed back
    by `close()`.  The history length D = `model.diffdel.max_delay` must fit the on-chip ring: D <= 32639 for one stream,
    16255 for two, 8063 for three or four.  The delay assert (`model.diffdel.check_delay`, read at open) runs on the host
    copy of each block, without a device synchronisation; a refused block raises AssertionError and changes nothing.
    Tensor-core modes only.  While the stream is open do not synchronise the whole device: the resident kernel only ends
    at `close()` or after `idle_timeout_ms` without a block."""

    def __init__(self, model, n_streams=1, block_len=64, idle_timeout_ms=5000):
        super().__init__(model, n_streams, block_len, idle_timeout_ms)
        self._pre = torch.empty((self.B, self.T), dtype=torch.float32)
        self._fn = _lib.load().ntm_rt_diffdel_process
        self._pp = ctypes.c_void_p(self._pre.data_ptr())
        self.d_in = torch.zeros((self.B, self.T), dtype=torch.float32)       # optional fixed delay block for step()
        self._dp = ctypes.c_void_p(self.d_in.data_ptr())

    def _open(self, h_host, idle_timeout_ms):
        m = self.model
        self.D = int(m.diffdel.max_delay)
        hist_host = m.diffdel._history(self.B, self.device).reshape(self.B, self.D).to("cpu").contiguous()
        return _lib.load().ntm_rt_diffdel_open(m._handle(self.device), _lib.MODES[m.mode], _ptr(h_host), _ptr(hist_host),
                                               self.B, self.T, self.D, int(bool(m.skip)), int(bool(m.diffdel.check_delay)),
                                               idle_timeout_ms, ctypes.byref(self._rt))

    def step(self):
        """Lowest-overhead form: process the blocks the caller wrote into `self.x_in` / `self.d_in`; returns the internal
        (y, pre_d) blocks (overwritten by the next call)."""
        rc = self._fn(self._live(), self._xp, self._dp, self._yp, self._pp)
        if rc:
            _lib.check(rc)
        return self._y, self._pre

    def process(self, x, d):
        rt = self._live()
        xt, dt = self._host_block(x, "x"), self._host_block(d, "d")
        rc = self._fn(rt, ctypes.c_void_p(xt.data_ptr()), ctypes.c_void_p(dt.data_ptr()), self._yp, self._pp)
        if rc:
            _lib.check(rc)
        return self._y.reshape(xt.shape), self._pre.reshape(xt.shape)

    def _stop(self, h=None):
        """Stop the resident kernel; with `h` given, the final state goes into it and the rolled history back to the
        model (`model.diffdel.buffer`)."""
        hist = None if h is None else torch.empty((self.B, self.D), dtype=torch.float32)
        rt, self._rt = self._rt, None
        _lib.check(_lib.load().ntm_rt_diffdel_close(rt, _ptr(h), _ptr(hist)))
        if hist is not None:
            self.model.diffdel.buffer = hist.reshape(self.B, 1, self.D).to(self.device)

    def close(self):
        """Stop the resident kernel and hand the carried state and delay history back to the model (`model.hidden`,
        `model.diffdel.buffer`)."""
        return super().close(), self.model.diffdel.buffer
