"""optiml_b200 -- B200-native (sm_100a) implementation of OptiML's kernel-SVM dual training path.

Drop-in names (same modules as the reference package ``optiml``):
    optiml_b200.ml.svm            SVC, SVR, DualSVC, DualSVR
    optiml_b200.ml.svm.kernels    LinearKernel, PolyKernel, GaussianKernel, linear, poly, gaussian
    optiml_b200.ml.svm.losses     hinge, epsilon_insensitive (tags)
    optiml_b200.opti              Quadratic, Optimizer
    optiml_b200.opti.constrained  BoxConstrainedQuadraticOptimizer, ProjectedGradient, FrankWolfe, AugmentedLagrangianQuadratic
    optiml_b200.opti.unconstrained.stochastic   AdaGrad, Adam, ... on the augmented-Lagrangian dual
and, for the reference's multi-class recipe (sklearn's OneVsRestClassifier over SVC), drop-ins whose binary problems
share ONE Gram matrix in HBM:
    optiml_b200.ml.multiclass     OneVsRestClassifier, MultiOutputRegressor
and, for model selection over optimizer='smo' estimators, sklearn's searches with the (candidate, fold) problems on
shared Gram matrices:
    optiml_b200.model_selection   GridSearchCV, cross_validate, cross_val_score

All numerical work is done by hand-written CUDA kernels behind the C ABI in include/svmb200.h
(optiml_b200/_lib/libsvmb200.so, built by optiml_b200/csrc/build.py).  There is no CPU fallback.
"""
__version__ = '0.1.0'
