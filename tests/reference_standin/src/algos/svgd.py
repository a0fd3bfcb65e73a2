from src.algos.util import Unpatched


class SVGDOptimizer(Unpatched):
    pass


def rbf(*args, **kwargs):
    raise AssertionError("stand-in rbf called: install() did not rebind it")
