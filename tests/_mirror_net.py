"""A small stand-in with the reference Network's call surface (SURVEY.md section 8 N-0): the reference
itself does not travel to the GPU box, so the drop-in ``forward`` functions are exercised on this.

Same attributes/methods the replaced ``forward``s touch: ``maxdisp``, ``disp``,
``feature(img, task_arch, path)``, ``matching(cost, task_arch, path)``, ``search_feature(img, ops)``,
``search_matching(cost, ops, t)``; per-layer ``nn.ModuleList``s indexed by ``task_arch[name][0]`` like
rag_model.py:291-295,331-336."""
import torch
import torch.nn as nn


class MirrorNet(nn.Module):
    def __init__(self, disp_module, maxdisp=192, n_paths=2, c=12):
        super().__init__()
        self.maxdisp = maxdisp
        self.disp = disp_module
        self.stem2d = nn.ModuleList([nn.Conv2d(3, c, 3, stride=3, padding=0, bias=False) for _ in range(n_paths)])
        self.last2d = nn.ModuleList([nn.Conv2d(c, c, 1, bias=False) for _ in range(n_paths)])
        self.stem3d = nn.ModuleList([nn.Conv3d(2 * c, c, 3, padding=1, bias=False) for _ in range(n_paths)])
        self.last3d = nn.ModuleList([nn.Conv3d(c, 1, 3, padding=1, bias=False) for _ in range(n_paths)])

    @staticmethod
    def _pick(task_arch, name):
        return 0 if task_arch is None else task_arch[name][0]

    def feature(self, x, task_arch=None, path=None):
        x = torch.relu(self.stem2d[self._pick(task_arch, "stem2d")](x))
        return self.last2d[self._pick(task_arch, "last2d")](x)

    def matching(self, cost, task_arch=None, path=None):
        x = torch.relu(self.stem3d[self._pick(task_arch, "stem3d")](cost))
        return self.last3d[self._pick(task_arch, "last3d")](x)

    def search_feature(self, x, selected_ops):
        return self.feature(x, None)

    def search_matching(self, cost, selected_ops, t):
        return self.matching(cost, None)


def arch(i):
    return {"stem2d": [i], "last2d": [i], "stem3d": [i], "last3d": [i]}


def reference_modules():
    """Fresh stand-ins for the three reference modules that ``rag_b200.network.install()`` rebinds, with the names it
    touches: ``models.rag_model`` (``Network.forward`` / ``search_forward``, ``Disp``, ``DisparityRegression``, ``nn``),
    ``automl.mdenas_basicmodel`` (``BasicNetwork.forward``, ``Disp``, ``DisparityRegression``) and
    ``automl.operations_3d`` (``ConvBR_3d.forward``).  Only the bindings are real: the stand-in methods raise."""
    import types

    def unpatched(*args, **kwargs):
        raise NotImplementedError("stand-in of a reference method: only its binding exists")

    def cls(name, *methods):                    # a distinct function object per method, so a crossed restore is visible
        return type(name, (nn.Module,), {m: (lambda *a, **k: unpatched()) for m in methods})

    def module(name, **attrs):
        m = types.ModuleType(name)
        m.__dict__.update(attrs)
        return m

    rag_model = module("models.rag_model", nn=nn, Network=cls("Network", "forward", "search_forward"),
                       Disp=cls("Disp", "forward"), DisparityRegression=cls("DisparityRegression", "forward"))
    mdenas_basicmodel = module("automl.mdenas_basicmodel", BasicNetwork=cls("BasicNetwork", "forward"),
                               Disp=cls("Disp", "forward"), DisparityRegression=cls("DisparityRegression", "forward"))
    operations_3d = module("automl.operations_3d", ConvBR_3d=cls("ConvBR_3d", "forward"))
    return rag_model, mdenas_basicmodel, operations_3d
