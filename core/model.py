"""Model: network + loss + optimiser (interface of the reference's core/model.py).

step()/zero_grad() keep the reference semantics (model.py:45-68) on top of two flat device
arenas -- one for every parameter, one for every gradient, laid out in the reference's flatten
order (layers in order, `w` then `b`, optimizer.py:14-15):
  * zero_grad()  = flags only (a slot is overwritten by the first gradient of the step)
  * backward     = GEMM / column-sum kernels write parameter gradients straight into their slots
  * step()       = (data parallel: one NCCL all-reduce of the gradient arena) + one fused
                   optimiser kernel over the arenas
"""
import pickle

import numpy as np

import core._backend as be
import core._deferred as deferred
import core._dist as dist
import core.ops as ops
import core.tensor as T

_ALIGN = 64  # elements; keeps every parameter slot 256-byte aligned for 128-bit kernels / TMA


class Model(object):

    # train_step on a small Dense/ReLU MLP with SoftmaxCrossEntropyLoss (the examples/mnist network)
    # records the fused small-MLP pass (csrc/mlp_fused.cu) instead of the layer-by-layer step
    fuse_small_mlp = True
    # the five-line loop of run.py:78-83 reaches the recorded step on its own (core/_deferred.py) ...
    defer_loop = deferred.ENABLED
    # ... as the layer-by-layer recording (bit-identical to the eager lines); True lets it be the fused
    # small-MLP pass where that applies (rounding-level differences, see train_step)
    defer_loop_may_fuse = False
    # ... for launch-bound steps only: batch and parameter counts up to these many elements.  A wide
    # step gains nothing from a replay (measured: 7.91 vs 7.92 ms for the 4 x 4096 MLP) and its
    # recording would pin the step's temporaries
    defer_loop_max_batch_elems = 1 << 22
    defer_loop_max_param_elems = 1 << 23
    defer_loop_max_recordings = 8     # distinct batch shapes a loop may have recorded at a time

    def __init__(self, net, loss, optimizer):
        self.net = net
        self.loss = loss
        self.optimizer = optimizer
        self._phase = "TRAIN"
        self._arena = None  # dict(params=[...], p=DArray, g=DArray, slots=[(off, size)])
        self._captured = {}  # batch signature -> "warm" | _CapturedStep | "eager"
        self._out_sig = {}   # (input shape, dtype) -> (output shape, dtype) seen in TRAIN phase
        self._noloop = set() # input signatures whose iteration could not be recorded
        self._stash_pred = False
        self._last_pred = None

    def forward(self, inputs):
        if self.defer_loop and self._phase == "TRAIN" and type(inputs) is T.Tensor:
            sig = self._out_sig.get((inputs.shape, inputs.dtype.str))
            if sig is not None and self._loop_can_defer(inputs):
                return deferred.begin(self, inputs, sig[0], sig[1])
            out = self.net.forward(inputs)
            self._note_output(inputs, out)
            return out
        return self.net.forward(inputs)

    def _note_output(self, inputs, out):
        if type(out) is T.Tensor and out.requires_grad:
            self._out_sig[(inputs.shape, inputs.dtype.str)] = (out.shape, out.dtype)

    def _loop_can_defer(self, x):
        """is this forward() the second line of a run.py-style iteration that step() could replay?
        Parameters in their arena with freshly zeroed gradients (zero_grad() was the first line), a
        built-in update rule, an input that needs no gradient, and no earlier failure to record
        this batch shape."""
        if x.requires_grad or (x.shape, x.dtype.str) in self._noloop or not ops._GRAD_ENABLED:
            return False
        if x._data.size > self.defer_loop_max_batch_elems:
            return False
        opt = self.optimizer
        if not _builtin_rule(opt):
            return False
        plist = self._param_list()
        if not plist or not self._arena_valid(plist):
            return False
        if self._arena["p"].size > self.defer_loop_max_param_elems:
            return False
        for p in plist:
            if not (p._grad_zero and p._grad is p._gslot and p.requires_grad):
                return False
        return True

    def predict(self, inputs):
        """forward pass without an autograd graph (the evaluation at run.py:87-91): activations are
        released as soon as the next layer has consumed them.  Not in the reference's interface."""
        from core.tensor import Tensor
        x = inputs if isinstance(inputs, Tensor) else Tensor(inputs)
        with ops.no_grad():
            return self.net.forward(x)

    # ------------------------------------------------------------------ checkpoint (values only)
    def save(self, path):
        """one dict per layer: its parameters' values, then its buffers' (BatchNormalization's
        running statistics) under their own names"""
        state = []
        for layer, params in zip(self.net.layers, self.net.get_parameters()):
            entry = {k: v.values for k, v in params.items() if v is not None}
            entry.update((k, v.values) for k, v in getattr(layer, "buffers", {}).items())
            state.append(entry)
        with open(path, "wb") as f:
            pickle.dump(state, f, -1)
        print("Model saved in %s." % path)

    def load(self, path):
        with open(path, "rb") as f:
            state = pickle.load(f)
        if hasattr(state, "layers"):
            # a checkpoint in the reference's format (model.py:18-21 pickles the whole Net): its
            # tensors were unpickled without going through __init__ and carry the reference's
            # attribute names -- take the arrays out of them
            state = [{k: _pickled_values(v) for k, v in getattr(layer, "params", {}).items()
                      if v is not None} for layer in state.layers]
        params = self.net.get_parameters()
        if len(state) != len(params):
            raise ValueError("Incompatible architecture: %d layers in the file, %d in the model"
                             % (len(state), len(params)))
        for layer, saved in zip(self.net.layers, state):
            for k, arr in saved.items():
                buf = getattr(layer, "buffers", {}).get(k)
                if buf is not None:
                    # copied into the existing device array: a recorded step that names it stays valid
                    if tuple(buf.shape) != tuple(arr.shape):
                        raise ValueError("Incompatible architecture. %s in loaded model and %s in "
                                         "defined model." % (arr.shape, buf.shape))
                    be.upload_into(buf._data, arr)
                    buf._touch()
                    continue
                cur = layer.params.get(k)
                if cur is not None and tuple(cur.shape) != tuple(arr.shape):
                    raise ValueError("Incompatible architecture. %s in loaded model and %s in "
                                     "defined model." % (arr.shape, cur.shape))
                if cur is None:
                    from core.tensor import Tensor
                    layer.params[k] = Tensor(arr, requires_grad=True, dtype=arr.dtype)
                    if hasattr(layer, "is_init"):
                        layer.is_init = True
                    if hasattr(layer, "shapes") and k in layer.shapes:
                        layer.shapes[k] = list(arr.shape)
                else:
                    cur.values = arr
                    cur.zero_grad()
        self._arena = None
        print("Restored model from %s." % path)

    def get_phase(self):
        return self._phase

    def set_phase(self, phase):
        assert phase in ("TRAIN", "TEST")
        self.net.set_phase(phase)
        self._phase = phase

    # ------------------------------------------------------------------ arenas
    def _param_list(self):
        return [p for layer in self.net.get_parameters() for p in layer.values() if p is not None]

    def _arena_valid(self, plist):
        a = self._arena
        if a is None or len(a["params"]) != len(plist):
            return False
        for p, q, (off, size) in zip(plist, a["params"], a["slots"]):
            if p is not q or p._data.buf is not a["p"].buf or p._gslot is None:
                return False
            if p._data.ptr != a["p"].ptr + off * a["p"].dtype.itemsize:
                return False
        return True

    def _build_arena(self, plist):
        """move parameters and their gradients into flat arenas; False if they cannot share one"""
        if not plist:
            return False
        dt = plist[0].dtype
        if any(p.dtype != dt for p in plist):
            return False
        slots, off = [], 0
        for p in plist:
            slots.append((off, p._data.size))
            off += (p._data.size + _ALIGN - 1) // _ALIGN * _ALIGN
        pa = be.zeros((off,), dt)
        ga = be.zeros((off,), dt)
        for p, (o, size) in zip(plist, slots):
            view = pa.view(p.shape, o)
            be.copy_into(view, p._data)
            gview = ga.view(p.shape, o)
            had_grad = p._grad is not None and not p._grad_zero
            if had_grad:
                be.copy_into(gview, p._grad)
            was_unset = p._grad is None and not p._grad_zero
            p._data = view
            p._host = None
            p._gslot = gview
            if was_unset:
                p._grad, p._grad_zero = None, False
            else:
                p._grad, p._grad_zero = gview, not had_grad
            p._grad_host = None
        self._arena = dict(params=list(plist), p=pa, g=ga, slots=slots)
        for st in self._captured.values():   # recorded steps name the old parameter addresses
            if not isinstance(st, str):
                st.destroy()
        self._captured = {}
        return True

    # ------------------------------------------------------------------ training step
    def step(self):
        chain = T._DEFERRED[0]
        if chain is not None:
            T._DEFERRED[0] = None
            if chain.model is self and chain.stage == "backward" and self._deferred_step(chain):
                return
            chain.materialise()
        plist = self._param_list()
        # the fused arena kernel implements the built-in update rules only: an optimiser whose class
        # overrides the reference's extension points (_compute_step / compute_step) goes through
        # compute_step(), consistently from its first step on (its state then has the reference's
        # unpadded flat layout)
        fused = _builtin_rule(self.optimizer) and (
            self._arena_valid(plist) or self._build_arena(plist))
        if fused:
            for p in plist:
                # a gradient that lives outside its arena slot (user code assigned `p.grad = ...`):
                # bring it into the slot instead of leaving the fused path -- the optimiser state is
                # laid out over the padded arena and cannot follow to the unpadded generic layout
                if p._grad is not p._gslot:
                    if p._grad is None:
                        if not p._grad_zero:
                            raise TypeError("a parameter has no gradient (call zero_grad() first)")
                    else:
                        be.copy_into(p._gslot, p._coerce_grad(p._grad))
                        p._grad_zero = False
                    p._grad, p._grad_host = p._gslot, None
            a = self._arena
            for p in plist:
                if p._grad_zero:             # no gradient reached this parameter in this step
                    be.memset_zero(p._gslot)
            if dist.world_size() > 1:
                # SUM (1/m_global is already inside dL/dz), in chunks pipelined with the optimiser
                dist.reduce_and_apply(self.optimizer, a["p"], a["g"], _ALIGN)
            else:
                self.optimizer.apply_fused(a["p"], a["g"])
            for p in plist:
                p._touch()
                p._drop_grad()  # reference: `param += step` leaves grad = None (tensor.py:35-38)
            return
        self._step_generic()

    def _deferred_step(self, chain):
        """zero_grad / forward / loss / backward were postponed (core/_deferred.py) and this is the
        iteration's step(): replay the recording of this batch shape if there is one (made once the
        shape has been through one eager iteration).  False = run the postponed lines eagerly."""
        x, y, loss_obj = chain.x, chain.y, chain.loss_obj
        # the layer-by-layer recording: the same kernels in the same order as the eager lines, so
        # the loop's numbers do not depend on whether an iteration was replayed (the fused
        # small-MLP pass sums in another order and stays behind the explicit train_step)
        key = self._step_key(x, y, loss_obj, "loop-fused" if self.defer_loop_may_fuse else "loop")
        state = self._captured.get(key)
        if state is not None and not isinstance(state, str) and not self._arena_valid(self._param_list()):
            self._drop_recordings()
            state = None
        if state is None:
            # first sight of this shape: it runs as written; the next one is recorded
            self._captured[key] = "warm"
            return False
        if state == "eager":
            self._noloop.add((x.shape, x.dtype.str))
            return False
        if state == "warm":
            n_rec = sum(1 for k, st in self._captured.items()
                        if not isinstance(st, str) and k[0].startswith("loop"))
            if n_rec >= self.defer_loop_max_recordings:
                # a loop over ever-changing batch shapes: each recording pins its temporaries
                self._captured[key] = "eager"
                self._noloop.add((x.shape, x.dtype.str))
                return False
            state = self._capture_step(x, y, key, loss_obj, allow_fused=self.defer_loop_may_fuse)
            if state is None:
                self._captured[key] = "eager"
                self._noloop.add((x.shape, x.dtype.str))
                return False
            self._captured[key] = state
        deferred.pin_live_prediction(state)
        loss = state.run(x, y)
        deferred.serve_after_replay(chain, state, loss._data)
        return True

    def _drop_recordings(self):
        for st in self._captured.values():
            if not isinstance(st, str):
                st.destroy()
        self._captured = {}

    def _step_key(self, x, y, loss_obj, kind="train_step"):
        # (loss objects of one class without state are interchangeable: run.py:72-73 builds two)
        # the layer list is part of the key: swapping an activation leaves every parameter where it
        # was, but a recording of the old network must not be replayed for the new one
        key = (kind, x.shape, x.dtype.str, y.shape, y.dtype.str, dist.world_size(), id(self.optimizer),
               type(loss_obj), id(getattr(loss_obj, "_weight", None)), self._phase,
               tuple((id(layer), type(layer)) for layer in self.net.layers))
        # a loss with a fixed configuration (HuberLoss's delta) is interchangeable only with one
        # configured alike: a recording bakes the configuration into its kernels' arguments
        config = getattr(loss_obj, "_config", None)
        return key + (config(),) if config is not None else key

    def _step_generic(self):
        """the reference's three stages verbatim (model.py:45-61), on device arrays"""
        params = self.net.get_parameters()
        all_grads = []
        for param in params:
            grad = dict()
            for k in param:
                p = param[k]
                if p._grad_zero:
                    grad[k] = be.zeros(p.shape, p.dtype)
                else:
                    grad[k] = p._grad
                if grad[k] is None:
                    raise TypeError("parameter %r has no gradient (call zero_grad() first)" % k)
            all_grads.append(grad)
        if dist.world_size() > 1:
            for grad in all_grads:
                for g in grad.values():
                    dist.allreduce_sum(g)
        steps = self.optimizer.compute_step(all_grads, params)
        for step, param in zip(steps, params):
            for k in param:
                param[k] += step[k]

    # ------------------------------------------------------------------ whole step, captured
    def train_step(self, inputs, targets):
        """One iteration of the reference's training loop (run.py:78-83) as a single call:

            model.zero_grad(); pred = model.forward(inputs); loss = model.loss.loss(pred, targets)
            loss.backward(); model.step()

        and the loss Tensor is returned.  The first call with a given batch shape runs exactly those
        five lines; the second records them into a CUDA graph (every kernel, memset and NCCL
        collective of the step, with its temporaries at fixed addresses); later calls copy the
        batch into the graph's input buffers and replay it with one launch, which removes the
        per-kernel launch cost that bounds the MNIST-sized step.  Values are bit-identical to the
        eager step (tests/test_gpu_graph.py).  A replay does not refresh the per-layer `inputs`
        bookkeeping or non-leaf `.grad`s -- use the five lines above when those are wanted."""
        from core.tensor import Tensor
        T._flush_deferred()
        x = inputs if isinstance(inputs, Tensor) else Tensor(inputs)
        y = targets if isinstance(targets, Tensor) else Tensor(targets)
        key = self._step_key(x, y, self.loss)
        state = self._captured.get(key)
        if state is not None and not isinstance(state, str):
            # a recorded step names the parameter arenas: if a parameter was rebound since
            # (p.values = ..., load(), set_parameters) every recording is stale
            if not self._arena_valid(self._param_list()):
                self._drop_recordings()
                state = None
        if state is None or state == "eager":
            loss = self._eager_step(x, y)
            if state is None:
                # _build_arena (first step) clears the table, so set the mark afterwards
                self._captured[key] = "warm"
            return loss
        if state == "warm":
            state = self._capture_step(x, y, key)
            if state is None:
                self._captured[key] = "eager"
                return self._eager_step(x, y)
            self._captured[key] = state
        deferred.pin_live_prediction(state)
        return state.run(x, y)

    def _eager_step(self, x, y, loss_obj=None):
        self.zero_grad()
        pred = self.net.forward(x)
        if self._stash_pred:             # a recording keeps its prediction's buffers (core/_deferred.py)
            self._last_pred = pred
        loss = (loss_obj or self.loss).loss(pred, y)
        loss.backward()
        self.step()
        return loss

    def _capture_step(self, x, y, key, loss_obj=None, allow_fused=True):
        loss_obj = loss_obj or self.loss
        plist = self._param_list()
        if not (plist and self._arena_valid(plist)) or not _builtin_rule(self.optimizer):
            return None
        plan = self._fused_mlp_plan(x, y, loss_obj) if (self.fuse_small_mlp and allow_fused) else None
        if plan is not None:
            body = lambda xt, yt: self._fused_mlp_step(xt, yt, plan)
        else:
            body = lambda xt, yt: self._eager_step(xt, yt, loss_obj)
        self._stash_pred = plan is None
        try:
            step = _CapturedStep(self, x, y, body, keepalive=plan)
            if plan is not None:
                tail = plan["tail"]
                step.prediction_source = lambda: (tail.logits, tail.dlogits)
            else:
                pred = self._last_pred
                step.prediction_source = lambda: (pred._data, pred._grad)
        except be.BackendError:
            # something in the step cannot be recorded (a host read of a device value, an upload,
            # scratch growth): the aborted recording ran nothing, so drop what it cached and let the
            # caller run this batch -- and every later one of this shape -- eagerly
            be.new_split_epoch()
            for p in plist:
                p._touch()
            self.zero_grad()
            return None
        finally:
            self._stash_pred, self._last_pred = False, None
        if not self._arena_valid(plist):   # the recorded step left the fused path
            step.destroy()
            return None
        return step

    # ------------------------------------------------------------------ fused small-MLP step
    def _fused_mlp_plan(self, x, y, loss_obj=None):
        """Is this (network, loss, batch) the pattern csrc/mlp_fused.cu handles?  A Dense/ReLU stack
        of float32 layers (run.py:59-69) whose layers after the first fit one SM's shared memory,
        the reference's SoftmaxCrossEntropyLoss, one process.  Returns the plan or None."""
        from core.layers import Dense, ReLU
        from core.losses import SoftmaxCrossEntropyLoss
        layers = self.net.layers
        loss_obj = loss_obj or self.loss
        if dist.world_size() != 1 or type(loss_obj) is not SoftmaxCrossEntropyLoss:
            return None
        if getattr(loss_obj, "_weight", None) is not None:
            return None
        if len(layers) < 3 or len(layers) % 2 == 0:
            return None
        dense = layers[0::2]
        if not all(type(l) is Dense and l.is_init for l in dense) or not all(type(l) is ReLU for l in layers[1::2]):
            return None
        plist = self._param_list()
        a = self._arena
        if a is None or not self._arena_valid(plist) or len(plist) != 2 * len(dense) or a["p"].dtype != be.F32:
            return None
        if x.dtype != be.F32 or x.ndim != 2 or y.ndim != 2 or y.dtype not in (be.F32, be.F64):
            return None
        dims = [dense[0].params["w"].shape[1]] + [l.params["w"].shape[1] for l in dense[1:]]
        B = x.shape[0]
        if x.shape[1] != dense[0].params["w"].shape[0] or y.shape != (B, dims[-1]):
            return None
        for l, d_in, d_out in zip(dense[1:], dims[:-1], dims[1:]):
            if tuple(l.params["w"].shape) != (d_in, d_out) or tuple(l.params["b"].shape) != (1, d_out):
                return None
        if tuple(dense[0].params["b"].shape) != (1, dims[0]) or not be.MLPTail.eligible(dims, B):
            return None
        n_grad = a["g"].size - a["slots"][2][0]
        return dict(dense=dense, dims=dims, tail=be.MLPTail(dims, B, n_grad))

    def _fused_mlp_step(self, x, y, plan):
        """zero_grad + forward + loss + backward + step of run.py:79-83 as: first-layer product,
        the fused tail pass, first-layer gradient products, optimiser.  Returns the loss Tensor."""
        from core.tensor import Tensor
        a, dense, dims = self._arena, plan["dense"], plan["dims"]
        be.new_split_epoch()
        w1, b1 = dense[0].params["w"], dense[0].params["b"]
        xd = x._data
        B = xd.shape[0]
        z1 = be.matmul(xd, w1._data, bias=b1._data)
        off_tail = a["slots"][2][0]
        n_grad = a["g"].size - off_tail
        offsets = [o - off_tail for (o, _) in a["slots"][2:]]
        dz1 = be.empty((B, dims[0]), be.F32)
        loss = be.empty((), be.F32)
        plan["tail"].run([l.params["w"]._data for l in dense[1:]], [l.params["b"]._data for l in dense[1:]],
                         a["g"].view((n_grad,), off_tail), offsets, n_grad, z1, y._data, B, dz1, loss)
        if be.dense_bwd_grouped_ok(B, w1.shape[0], w1.shape[1], be.F32):
            be.dense_bwd_grouped(dz1, xd, w1._data, None, False, w1._gslot, False, b1._gslot, False)
        else:
            be.matmul(xd, dz1, ta=True, out=w1._gslot)
            be.colsum(dz1, out=b1._gslot)
        self.optimizer.apply_fused(a["p"], a["g"])
        for p in a["params"]:
            p._touch()
            p._drop_grad()
        return Tensor(loss)

    def zero_grad(self):
        chain = T._DEFERRED[0]
        if chain is not None and chain.stage == "backward":
            T._flush_deferred()          # a postponed backward() has gradients to leave behind first
        be.new_split_epoch()
        plist = self._param_list()
        if plist and self._arena_valid(plist):
            # no memset of the arena: the backward pass overwrites every slot it reaches (the first
            # write of a step does not accumulate) and step() clears the ones it did not reach
            for p in plist:
                p._grad, p._grad_zero, p._grad_host = p._gslot, True, None
            return
        for p in plist:
            p.zero_grad()


def _builtin_rule(opt):
    """one of core/optimizer.py's fused update rules, not overridden -- False also for an optimiser
    object that merely offers the reference's compute_step() (model.py:55) without deriving from
    BaseOptimizer"""
    check = getattr(opt, "uses_builtin_rule", None)
    return getattr(opt, "opt_code", None) is not None and check is not None and bool(check())


def _pickled_values(t):
    """the ndarray inside a tensor that came out of pickle: this engine's Tensor, or the
    reference's (attribute `_values`, tensor.py:20), or a bare array"""
    if isinstance(t, np.ndarray):
        return t
    d = getattr(t, "__dict__", {})
    if "_values" in d:
        return np.asarray(d["_values"])
    if "_data" in d or hasattr(t, "values"):
        return np.asarray(t.values)
    raise ValueError("unrecognised checkpoint entry of type %s" % type(t).__name__)


class _CapturedStep(object):
    """The training step of one batch shape, recorded once and replayed (Model.train_step)."""

    def __init__(self, model, x, y, body=None, keepalive=None):
        """body(x_tensor, y_tensor) -> loss Tensor is what gets recorded (default: the five lines);
        keepalive: whatever owns device buffers the recording names besides its own temporaries"""
        from core.tensor import Tensor
        self.model = model
        self.keepalive = keepalive
        body = body or model._eager_step
        self.x = be.empty(x.shape, x.dtype)          # the graph reads its batch from here
        self.y = be.empty(y.shape, y.dtype)
        self.hyper = be.zeros((8,), be.F64)
        self.plist = model._param_list()
        self.layers = list(model.net.layers)   # kept alive: their ids are part of the recording's key
        opt = model.optimizer
        self.graph = be.StepGraph()
        for dt in (be.F32, be.F64):
            be.ones_scalar(dt)       # shared constants must exist (and hold 1.0) before recording
        opt._hyper_dev = self.hyper
        try:
            with self.graph.capture():
                loss = body(Tensor(self.x), Tensor(self.y))
                self.loss = loss._data                # stays allocated: the graph writes it
        finally:
            opt._hyper_dev = None
        # nothing ran: whatever the recording cached (host copies, tf32 planes) is not real
        be.new_split_epoch()
        for p in self.plist:
            p._touch()

    def run(self, x, y):
        from core.tensor import Tensor
        for dst, src in ((self.x, x._data), (self.y, y._data)):
            if isinstance(src, be.LazyRows) and src._real is None:
                src.gather_into(dst)        # rows perm[start:end] straight into the graph's input
            elif isinstance(src, be.LazyOneHot) and src._real is None:
                # class indices -> one-hot rows written straight into the graph's label buffer
                be.one_hot_into(dst, src.labels_ptr, src.shape[0], src.shape[1])
            else:
                be.copy_into(dst, src)
        self.model.optimizer.upload_hyper(self.hyper)
        self.graph.replay()
        for p in self.plist:
            p._touch()
            p._drop_grad()   # as after the eager step(): `param += step` leaves grad = None (tensor.py:35-38)
        for layer in self.layers:
            for buf in getattr(layer, "buffers", {}).values():
                buf._touch()     # updated in place by the replay (running statistics)
        # the loss buffer is rewritten by the next replay: hand out a copy
        return Tensor(be.clone(self.loss))

    def info(self):
        return self.graph.info()

    def destroy(self):
        self.graph.destroy()
