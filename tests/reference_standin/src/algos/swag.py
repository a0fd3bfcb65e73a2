from src.algos.util import Unpatched


class SwagOptimizer(Unpatched):
    pass
