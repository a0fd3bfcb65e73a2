from src.algos.util import Unpatched


class LastLayerBayesianOptimizer(Unpatched):
    pass
