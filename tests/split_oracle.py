"""The CPU oracle (oracle/ref_graph.GraphExecutor) for graphs that contain ONNX Split.

Each Split node is replaced, after parsing, by one single-output "SplitPart" node per named output, which the executor's
node loop (run and run_forced alike) evaluates like any other op: output k of a Split is the k-th channel range of its
input, with the sizes from the `split` attribute (opset < 13), the `split` input (opset >= 13) or equal parts.  A part is
taken exactly from the tensor the executor holds for the input, so under run_forced it reads the forced tensor."""
import torch

from oracle import onnx_min, ref_graph


class SplitExecutor(ref_graph.GraphExecutor):
    def __init__(self, onnx_bytes: bytes, *args, **kwargs):
        super().__init__(onnx_bytes, *args, **kwargs)
        nodes = []
        for n in self.graph.nodes:
            if n.op != "Split":
                nodes.append(n)
                continue
            for k, out in enumerate(n.outputs):
                if out:
                    nodes.append(onnx_min.Node("SplitPart", f"{n.name}:{k}", list(n.inputs), [out],
                                               dict(n.attrs, index=k, parts=len(n.outputs))))
        self.graph.nodes = nodes

    def _node(self, n, ins, acc64: bool):
        if n.op != "SplitPart":
            return super()._node(n, ins, acc64)
        axis = n.attrs.get("axis", 0)
        if "split" in n.attrs:
            sizes = [int(v) for v in n.attrs["split"]]
        elif len(ins) > 1 and ins[1] is not None:
            sizes = [int(v) for v in ins[1]]
        else:
            sizes = [ins[0].shape[axis] // n.attrs["parts"]] * n.attrs["parts"]
        return torch.split(ins[0], sizes, dim=axis)[n.attrs["index"]]
