"""Autograd bridge shared by the drop-in modules: forward/backward of a whole network through a UNetEngine."""
import threading

import torch


class EngineFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, module, x, *params):
        engine = module._engine_for(x.device)
        names = module._param_names
        tensors = dict(zip(names, params))
        tensors.update(module._named_buffer_tensors())        # BatchNorm running statistics (updated in place)
        needs = any(ctx.needs_input_grad[2:])
        input_grad = ctx.needs_input_grad[1]          # x.grad: saliency maps, adversarial inputs, trainable modules in front
        trainable = {n for n, need in zip(names, ctx.needs_input_grad[2:]) if need}
        if needs or module.training:
            # parameters of a training module change between calls (optimizer steps, and in-place `.data` writes such as
            # weights_init / EMA that do not bump Tensor._version): always re-pack the bf16 operands (one launch)
            engine.invalidate_packed_weights()
        save = needs or input_grad
        logits = engine.forward(x, tensors, save=save, training=module.training, trainable=trainable, input_grad=input_grad)
        if save:
            engine._generation = getattr(engine, "_generation", 0) + 1
            ctx.generation = engine._generation
            ctx.engine = engine
            ctx.names = names
            ctx.params = params
            ctx.tensors = tensors
            ctx.x_meta = (x.shape, x.dtype)
        return logits

    @staticmethod
    def backward(ctx, dlogits):
        engine = ctx.engine
        if engine._generation != ctx.generation:
            raise RuntimeError("backward: the saved activations were overwritten by a later training forward")
        # zero-initialised: a gradient the engine legitimately leaves untouched (a tensor that cannot receive one) reads as
        # 0, never as uninitialised memory
        grads = {n: torch.zeros_like(p) for n, p, need in zip(ctx.names, ctx.params, ctx.needs_input_grad[2:]) if need}
        dx = None
        if ctx.needs_input_grad[1]:
            shape, dtype = ctx.x_meta
            dx = torch.empty(shape, dtype=torch.float32, device=dlogits.device)
        engine.backward(dlogits, ctx.tensors, grads, dx=dx)
        if dx is not None and dtype != torch.float32:
            dx = dx.to(dtype)
        return (None, dx) + tuple(grads.get(n) for n in ctx.names)


class EngineModuleMixin:
    """Gives an nn.Module (a pure parameter container) a forward() that runs on the CUDA engine.  One engine per
    device: nn.DataParallel replicas share this object's dict, each device thread gets its own engine."""

    def _make_engine(self, device):
        raise NotImplementedError

    def _engine_for(self, device):
        key = (device.type, device.index)
        with self._engine_lock:
            eng = self._engines.get(key)
            if eng is None:
                eng = self._make_engine(device)
                self._engines[key] = eng
            return eng

    def _init_engine_state(self):
        self._engines = {}
        self._engine_lock = threading.Lock()
        # names are fixed at construction: nn.DataParallel replicas carry their parameters as plain tensor attributes
        # (named_parameters() is empty there), so tensors are always fetched by walking the module tree by name
        self._pnames = [n for n, _ in self.named_parameters()]
        self._bnames = [n for n, _ in self.named_buffers()]
        self.register_load_state_dict_post_hook(lambda module, incompatible_keys: module.invalidate())

    @property
    def _param_names(self):
        return self._pnames

    def _by_name(self, name):
        obj = self
        for part in name.split("."):
            obj = getattr(obj, part)
        return obj

    def _named_buffer_tensors(self):
        return {n: self._by_name(n) for n in self._bnames}

    def invalidate(self):
        """Call after changing parameters of an eval-mode module behind autograd's back (`p.data` writes): the engines
        then re-pack their bf16 operands on the next forward.  load_state_dict does it by itself."""
        for eng in self._engines.values():
            eng.invalidate_packed_weights()

    def _engine_forward(self, inputs):
        if not inputs.is_cuda:
            raise RuntimeError(f"unet_pytorch_b200.{type(self).__name__} runs on a B200 only: move the module and inputs "
                               "to CUDA (there is no CPU fallback)")
        params = [self._by_name(n) for n in self._pnames]
        return EngineFunction.apply(self, inputs, *params)
