from src.algos.util import Unpatched


class BBBOptimizer(Unpatched):
    pass


class GaussianPrior(Unpatched):
    pass


class MixturePrior(Unpatched):
    pass
