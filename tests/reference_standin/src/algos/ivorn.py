from src.algos.util import Unpatched


class iVONOptimizer(Unpatched):
    pass
