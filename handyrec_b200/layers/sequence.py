"""Sequence layers (mirror of /root/reference/handyrec/layers/sequence.py:7-143)."""
from __future__ import annotations

import torch

from .._lib import HRB_UNSUPPORTED, HrbError
from ..autograd_ops import TC_MIN_ROWS, AttInputFn, LAUFirstLayerFn, MaskScoresFn, SeqPoolFn
from ..keras_lite import Layer
from .core import DNN


class SequencePoolingLayer(Layer):
    """Masked mean / max / sum pooling over axis 1 (sequence.py:26-46)."""

    def __init__(self, method: str, **kwargs):
        super().__init__(**kwargs)
        assert method in ["mean", "max", "sum"], "Pooling method should be `mean`, `max`, or `sum`"
        self.method = method

    def call(self, inputs, mask=None):
        if mask is None:
            raise ValueError("Embedding layer should set `mask_zero` as True")
        return SeqPoolFn.apply(inputs, mask, self.method)

    def compute_output_shape(self, input_shape):
        return (None, 1, input_shape[-1])

    def get_config(self):
        return {"method": self.method, **super().get_config()}


class LocalActivationUnit(Layer):
    """The LocalActivationUnit used in DIN (sequence.py:57-143)."""

    def __init__(self, hidden_units=(64, 32, 1), activation="sigmoid", l2_reg=0, dropout_rate=0, use_bn=False, seed=1024, **kwargs):
        self.hidden_units, self.activation, self.l2_reg = hidden_units, activation, l2_reg
        self.dropout_rate, self.use_bn, self.seed = dropout_rate, use_bn, seed
        self.dnn = None
        super().__init__(**kwargs)

    def build(self, input_shape):
        self._input_check(input_shape)
        self.dnn = self._track(DNN(self.hidden_units, self.activation, self.l2_reg, self.dropout_rate, self.use_bn, seed=self.seed))
        d = input_shape[0][-1]
        self.dnn.build((None, input_shape[1][1], 4 * d))
        self.built = True

    def _fused_inference(self, query, keys):
        """Inference (no gradient, moving Dice statistics): hrb_lau_fwd gathers q and the T keys from the table, builds
        [q,k,q-k,q*k] per tile in shared memory, runs the MLP, masks padded positions -- the (B,T,4D) tensor never exists."""
        from .. import kernels as K
        from .activation import Dice
        from .core import Dense

        src_q, src_k = getattr(query, "_hrb_src", None), getattr(keys, "_hrb_src", None)
        dnn = self.dnn
        if src_q is None or src_k is None or src_q[0].data_ptr() != src_k[0].data_ptr() or dnn.use_bn or torch.is_grad_enabled():
            return None
        if dnn.activation not in ("dice", "relu", "sigmoid", "tanh", "linear", None) or dnn.output_activation not in (None, "linear"):
            return None
        dense = [l for l in dnn.layers if isinstance(l, Dense)]
        dices = [l for l in dnn.layers if isinstance(l, Dice)]
        if dnn.activation == "dice" and len(dices) != len(dense) - 1:
            return None
        stats = [(d.alphas.data, d.moving_mean.data, d.moving_variance.data) for d in dices] if dnn.activation == "dice" else None
        params = K.lau_pack_params([d.kernel.data for d in dense], [d.bias.data for d in dense], stats)
        table, q_ids = src_q
        _, k_ids = src_k
        try:
            score, _ = K.lau_fwd(table, q_ids.reshape(-1).contiguous(), k_ids.contiguous(), params, [d.units for d in dense],
                                 dnn.activation or "linear", want_pooled=False)
        except HrbError as e:
            # widths the fused kernel cannot hold in shared memory (4D or a hidden layer of about 400 and more) are declared
            # unsupported before anything is launched; the layer-by-layer path computes the same scores
            if e.status != HRB_UNSUPPORTED:
                raise
            return None
        return score

    def call(self, inputs, mask=None, **kwargs):
        query, keys = inputs  # (?, 1, D), (?, T, D)
        key_mask = mask[1]    # (?, T) after SqueezeMask
        if not kwargs.get("training", False):
            fused = self._fused_inference(query, keys)
            if fused is not None:
                return fused
        B, T, D = keys.shape
        training = kwargs.get("training", False)
        first = self.dnn.layers[0]  # Dense(4D): core.py:57 prepends the input width to the hidden units
        if B * T >= TC_MIN_ROWS and D % 4 == 0 and 2 * D >= 16 and first.units % 4 == 0 and first.units >= 16 and first.use_bias and \
                first.activation in (None, "linear", "relu", "sigmoid", "tanh"):
            # tall input (DIN: B*T = 204 800 rows): the first layer runs as q-term + [k | q*k] GEMM on the tensor cores and the
            # (B,T,4D) tensor of sequence.py:96-97 is never built; the remaining layers follow as usual
            x = LAUFirstLayerFn.apply(query.reshape(B, D), keys, first.kernel, first.bias, first.activation)
            for l in self.dnn.layers[1:]:
                x = l.call(x, training=training) if l._call_takes_training else l.call(x)
            att_out = x
        else:
            att_input = AttInputFn.apply(query.reshape(B, D), keys)              # sequence.py:96-97
            att_out = self.dnn(att_input, training=training)                      # (?, T, 1)
        att_out = MaskScoresFn.apply(att_out.reshape(B, T), key_mask)             # sequence.py:100-101
        return att_out.reshape(B, 1, T)

    def compute_output_shape(self, input_shape):
        return input_shape[1][0], 1, input_shape[1][1]

    def compute_mask(self, inputs, mask):
        return mask

    def get_config(self):
        return {"activation": self.activation, "hidden_units": self.hidden_units, "l2_reg": self.l2_reg, "dropout_rate": self.dropout_rate,
                "use_bn": self.use_bn, "seed": self.seed, **super().get_config()}

    @staticmethod
    def _input_check(input_shape):
        if not isinstance(input_shape, list) or len(input_shape) != 2:
            raise ValueError("A `LocalActivationUnit` layer should be called on a list of 2 inputs")
        if len(input_shape[0]) != 3 or len(input_shape[1]) != 3:
            raise ValueError("Unexpected inputs dimensions %d and %d, expect to be 3 dimensions" % (len(input_shape[0]), len(input_shape[1])))
        if input_shape[0][-1] != input_shape[1][-1] or input_shape[0][1] != 1:
            raise ValueError("A `LocalActivationUnit` layer requires inputs of a two inputs with shape (None,1,embedding_size) and "
                             "(None,T,embedding_size) Got different shapes: %s,%s" % (input_shape[0], input_shape[1]))
