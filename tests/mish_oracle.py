"""The CPU oracle (oracle/ref_graph.GraphExecutor) for graphs with Mish, x * tanh(softplus(x)).

After parsing, every Mish is folded into one node: an ONNX `Mish` node, or the `Softplus -> Tanh -> Mul(x, tanh)` chain
torch's exporter writes for nn.Mish.  The folded node is an `Identity` marked `mish`, which this executor's node loop (run
and run_forced alike) evaluates as Mish, in the dtype of the pass (float64 under run_forced).  Being an Identity, it carries
S, the magnitude behind each element, through run_forced like LeakyRelu does.  In bf16 mode the value after the Mish is the
stored (rounded) activation, as the fused convolution stores it, and not the convolution's own output.  run_forced tags the
record of every value the Mish is fused into (the Mish output, and a residual Add / Resize / MaxPool that is the sole reader
of it) with rec["act"] = "mish", which selects the Mish form of the rounding model (tests/mish_compare.py)."""
import torch

from oracle import onnx_min, ref_graph


def mish(x: torch.Tensor) -> torch.Tensor:
    return x * torch.tanh(torch.logaddexp(x, torch.zeros_like(x)))


class MishExecutor(ref_graph.GraphExecutor):
    def __init__(self, onnx_bytes: bytes, *args, **kwargs):
        super().__init__(onnx_bytes, *args, **kwargs)
        self._fold_mish()  # (bf16 mode folded it already, before its rounding plan)
        readers = {}
        for n in self.graph.nodes:
            for i in n.inputs:
                readers.setdefault(i, []).append(n)
        self.mish_values = set()
        for n in self.graph.nodes:
            if n.attrs.get("mish"):
                name = n.outputs[0]
                while True:
                    self.mish_values.add(name)
                    r = readers.get(name, [])
                    if len(r) != 1 or r[0].op not in ("Add", "Resize", "Upsample", "MaxPool") or name in self.graph.outputs:
                        break
                    name = r[0].outputs[0]

    def _fold_mish(self):
        if getattr(self, "_folded_mish", False):
            return
        self._folded_mish = True
        g = self.graph
        producer = {o: n for n in g.nodes for o in n.outputs}
        drop, nodes = set(), []
        for n in g.nodes:
            if n.op == "Mish":
                nodes.append(onnx_min.Node("Identity", n.name, [n.inputs[0]], list(n.outputs), {"mish": 1}))
                continue
            if n.op == "Mul":
                for t in (0, 1):
                    th = producer.get(n.inputs[t])
                    sp = producer.get(th.inputs[0]) if th is not None and th.op == "Tanh" else None
                    if sp is not None and sp.op == "Softplus" and sp.inputs[0] == n.inputs[1 - t]:
                        drop.update((id(th), id(sp)))
                        n = onnx_min.Node("Identity", n.name, [sp.inputs[0]], list(n.outputs), {"mish": 1})
                        break
            nodes.append(n)
        g.nodes = [n for n in nodes if id(n) not in drop]

    def _prepare_bf16(self):
        self._fold_mish()
        super()._prepare_bf16()
        # the fused convolution stores the value after the Mish, not the convolution's output that feeds it
        for n in self.graph.nodes:
            if n.attrs.get("mish") and n.inputs[0] in self.round_after:
                self.round_after.discard(n.inputs[0])
                if n.outputs[0] not in self.graph.outputs:
                    self.round_after.add(n.outputs[0])

    def _node(self, n, ins, acc64: bool):
        if n.op == "Identity" and n.attrs.get("mish"):
            return mish(ins[0])
        if n.op == "Softplus":
            return torch.logaddexp(ins[0], torch.zeros_like(ins[0]))
        if n.op == "Tanh":
            return torch.tanh(ins[0])
        return super()._node(n, ins, acc64)

    def run_forced(self, x, overrides, on_value=None):
        def tag(name, rec):
            if name in self.mish_values:
                rec["act"] = "mish"
            return rec
        if on_value is not None:
            return super().run_forced(x, overrides, on_value=lambda name, rec: on_value(name, tag(name, rec)))
        recs = super().run_forced(x, overrides)
        for name, rec in recs.items():
            tag(name, rec)
        return recs
