"""The CPU-runnable cases of the reference's own test suite (jfkirk/tensorrec, test/), restated against this package the
way code written for the reference reaches it: `import tensorrec` and `import tensorflow` resolve to compat/.  Each case
is named by the reference test it restates; the known answers it compares against are the reference's own
(tests/golden/reference_known_answers.json).  Run with compat/ and the repository root on PYTHONPATH:

    PYTHONPATH=compat:. python -m tests.reference_cases test_loss_graphs.py

prints `PASS <case>` / `FAIL <case>` lines and exits non-zero if any case fails (tests/test_reference_suite_cpu.py)."""
import json
import os
import shutil
import sys
import tempfile
import traceback

import numpy as np

import tensorflow as tf
import tensorrec
from tensorrec import TensorRec
from tensorrec import loss_graphs as LG, prediction_graphs as PG, representation_graphs as RG
from tensorrec.errors import ModelNotFitException, BatchNonSparseInputException
from tensorrec.input_utils import create_tensorrec_dataset_from_sparse_matrix, write_tfrecord_from_sparse_matrix
from tensorrec.recommendation_graphs import (
    project_biases, split_sparse_tensor_indices, bias_prediction_serial, densify_sampled_item_predictions
)
from tensorrec.session_management import get_session, set_session
from tensorrec.util import calculate_batched_alpha, generate_dummy_data, generate_dummy_data_with_indicator

GOLDEN = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden',
                                     'reference_known_answers.json')))
CASES = {}


def case(target, name):
    def register(fn):
        CASES.setdefault(target, []).append((name, fn))
        return fn
    return register


def raises(exc, fn, *args, **kwargs):
    try:
        fn(*args, **kwargs)
    except exc:
        return
    raise AssertionError('%s did not raise %s' % (getattr(fn, '__name__', fn), exc.__name__))


def sparse_tensor(rows):
    m = np.array(rows, dtype=np.float32)
    r, c = np.nonzero(m)
    return tf.SparseTensor(np.stack([r, c], axis=1), m[r, c], m.shape)


# ---- test_util.py -----------------------------------------------------------------------------------------------
@case('test_util.py', 'UtilTestcase::test_calculate_batched_alpha')
def _batched_alpha():
    g = GOLDEN['calculate_batched_alpha']
    assert calculate_batched_alpha(num_batches=1, alpha=g['alpha']) == g['alpha']
    got = calculate_batched_alpha(num_batches=g['num_batches'], alpha=g['alpha'])
    assert round(got - g['expected_ratio'] * g['alpha'], 5) == 0
    raises(ValueError, calculate_batched_alpha, num_batches=0, alpha=g['alpha'])


# ---- test_loss_graphs.py: fit with every loss graph, biased or not ----------------------------------------------
def _fit_with_loss(graph, biased, sampled):
    def run():
        data = generate_dummy_data_with_indicator(num_users=10, num_items=12, interaction_density=.5)
        model = TensorRec(loss_graph=graph(), biased=biased) if biased else TensorRec(loss_graph=graph())
        model.fit(*data, epochs=5, **({'n_sampled_items': 10} if sampled else {}))
    return run


for _name, _graph, _sampled in (('rmse_loss', LG.RMSELossGraph, False), ('rmse_dense_loss', LG.RMSEDenseLossGraph, False),
                                ('wmrb_loss', LG.WMRBLossGraph, True),
                                ('balanced_wmrb_loss', LG.BalancedWMRBLossGraph, True)):
    for _biased in (False, True):
        case('test_loss_graphs.py', 'LossGraphsTestCase::test_%s%s' % (_name, '_biased' if _biased else ''))(
            _fit_with_loss(_graph, _biased, _sampled))


# ---- test_representation_graphs.py ------------------------------------------------------------------------------
def _repr_data(n_user_features, n_item_features):
    return generate_dummy_data(num_users=15, num_items=30, interaction_density=.5, num_user_features=n_user_features,
                               num_item_features=n_item_features, n_features_per_user=20, n_features_per_item=20,
                               pos_int_ratio=.5)


def _fit_with_repr(user_repr, item_repr, n_user_features, n_item_features, n_components):
    def run():
        model = TensorRec(n_components=n_components, user_repr_graph=user_repr(), item_repr_graph=item_repr())
        model.fit(*_repr_data(n_user_features, n_item_features), epochs=10)
        assert model.tf_prediction is not None
    return run


for _i, (_name, _u, _it, _nu, _ni, _nc) in enumerate((
        ('linear', RG.LinearRepresentationGraph, RG.LinearRepresentationGraph, 50, 60, 20),
        ('norm_lin', RG.NormalizedLinearRepresentationGraph, RG.NormalizedLinearRepresentationGraph, 50, 60, 20),
        ('fpt_user', RG.FeaturePassThroughRepresentationGraph, RG.NormalizedLinearRepresentationGraph, 50, 60, 50),
        ('fpt_item', RG.NormalizedLinearRepresentationGraph, RG.FeaturePassThroughRepresentationGraph, 50, 60, 60),
        ('fpt_both', RG.FeaturePassThroughRepresentationGraph, RG.FeaturePassThroughRepresentationGraph, 50, 50, 50),
        ('weighted_fpt', RG.WeightedFeaturePassThroughRepresentationGraph,
         RG.WeightedFeaturePassThroughRepresentationGraph, 50, 50, 50),
        ('relu', RG.ReLURepresentationGraph, RG.ReLURepresentationGraph, 50, 60, 20))):
    case('test_representation_graphs.py', 'RepresentationGraphTestCase::test_fit_%d_%s' % (_i, _name))(
        _fit_with_repr(_u, _it, _nu, _ni, _nc))


@case('test_representation_graphs.py', 'IdentityRepresentationGraphTestCase::test_fit_fail_on_bad_dims')
def _pass_through_width_mismatch():
    data = _repr_data(30, 20)
    for user_repr, item_repr in ((RG.FeaturePassThroughRepresentationGraph, RG.LinearRepresentationGraph),
                                 (RG.LinearRepresentationGraph, RG.FeaturePassThroughRepresentationGraph)):
        model = TensorRec(n_components=25, user_repr_graph=user_repr(), item_repr_graph=item_repr())
        raises(ValueError, model.fit, *data, epochs=10)


# ---- test_tensorrec.py::TensorRecTestCase -----------------------------------------------------------------------
class _TensorRecData(object):
    """15 users x 30 items, 200 user / 150 item features, and the same three matrices as TFRecord files."""
    ready = False

    @classmethod
    def get(cls):
        if not cls.ready:
            cls.interactions, cls.uf, cls.itf = generate_dummy_data(
                num_users=15, num_items=30, interaction_density=.5, num_user_features=200, num_item_features=150,
                n_features_per_user=20, n_features_per_item=20, pos_int_ratio=.5)
            set_session(None)
            cls.tmp = tempfile.mkdtemp()
            cls.paths = [os.path.join(cls.tmp, n + '.tfrecord') for n in ('interactions', 'user_features',
                                                                            'item_features')]
            for path, m in zip(cls.paths, (cls.interactions, cls.uf, cls.itf)):
                write_tfrecord_from_sparse_matrix(path, m)
            cls.ready = True
        return cls


def _tr(name):
    return case('test_tensorrec.py::TensorRecTestCase', 'TensorRecTestCase::' + name)


@_tr('test_init')
def _init():
    assert TensorRec() is not None


@_tr('test_init_fail_0_components')
def _init_0_components():
    raises(ValueError, TensorRec, n_components=0)


@_tr('test_init_fail_none_factory')
def _init_none_factory():
    for key in ('user_repr_graph', 'item_repr_graph', 'loss_graph'):
        raises(ValueError, TensorRec, **{key: None})


@_tr('test_init_fail_bad_loss_graph')
def _init_bad_loss():
    raises(ValueError, TensorRec, loss_graph=np.mean)


@_tr('test_init_fail_attention_with_1_taste')
def _init_attention_1_taste():
    raises(ValueError, TensorRec, n_tastes=1, attention_graph=RG.LinearRepresentationGraph())


@_tr('test_init_fail_bad_attention_graph')
def _init_bad_attention():
    raises(ValueError, TensorRec, attention_graph=np.mean)


@_tr('test_predict_fail_unfit')
def _predict_unfit():
    d = _TensorRecData.get()
    model = TensorRec()
    for call, args in ((model.predict, (d.uf, d.itf)), (model.predict_rank, (d.uf, d.itf)),
                       (model.predict_user_representation, (d.uf,)), (model.predict_item_representation, (d.itf,)),
                       (model.predict_user_attention_representation, (d.uf,)), (model.predict_item_bias, (d.itf,)),
                       (model.predict_user_bias, (d.uf,))):
        raises(ModelNotFitException, call, *args)
    raises(ModelNotFitException, model.predict_similar_items, d.itf, item_ids=[1], n_similar=5)


@_tr('test_fit_verbose')
def _fit_verbose():
    d = _TensorRecData.get()
    model = TensorRec(n_components=10)
    model.fit(d.interactions, d.uf, d.itf, epochs=10, verbose=True)
    assert model.tf_prediction is not None


@_tr('test_fit_batched')
def _fit_batched():
    d = _TensorRecData.get()
    model = TensorRec(n_components=10)
    model.fit(d.interactions, d.uf, d.itf, epochs=10, user_batch_size=2)
    assert model.tf_prediction is not None


@_tr('test_fit_fail_bad_input')
def _fit_bad_input():
    d = _TensorRecData.get()
    model = TensorRec(n_components=10)
    good = [d.interactions, d.uf, d.itf]
    for slot in range(3):
        args = list(good)
        args[slot] = np.array([1, 2, 3, 4])
        raises(ValueError, model.fit, *args, epochs=10)


@_tr('test_fit_fail_mismatched_batches')
def _fit_mismatched_batches():
    d = _TensorRecData.get()
    model = TensorRec(n_components=10)
    raises(ValueError, model.fit, d.interactions, [d.uf] * 2, [d.itf] * 3, epochs=10)
    raises(ValueError, model.fit, d.interactions, [d.uf] * 2, [d.itf] * 2, epochs=10)
    model.fit([d.interactions] * 2, [d.uf] * 2, d.itf, epochs=10)
    model.fit([d.interactions] * 2, [d.uf] * 2, [d.itf] * 2, epochs=10)


@_tr('test_fit_fail_batching_dataset')
def _fit_batching_dataset():
    d = _TensorRecData.get()
    model = TensorRec(n_components=10)
    raises(BatchNonSparseInputException, model.fit, create_tensorrec_dataset_from_sparse_matrix(d.interactions), d.uf,
           d.itf, epochs=10, user_batch_size=2)


def _fit_with_datasets(as_dataset):
    def run():
        d = _TensorRecData.get()
        args = [create_tensorrec_dataset_from_sparse_matrix(m) if flag else m
                for m, flag in zip((d.interactions, d.uf, d.itf), as_dataset)]
        TensorRec(n_components=10).fit(*args, epochs=10)
    return run


for _name, _flags in (('test_fit_user_feature_as_dataset', (False, True, False)),
                      ('test_fit_item_feature_as_dataset', (False, False, True)),
                      ('test_fit_interactions_as_dataset', (True, False, False)),
                      ('test_fit_from_datasets', (True, True, True))):
    _tr(_name)(_fit_with_datasets(_flags))


@_tr('test_fit_from_tfrecords')
def _fit_tfrecords():
    d = _TensorRecData.get()
    set_session(None)
    TensorRec(n_components=10).fit(*d.paths, epochs=10)


# ---- test_readme.py: user-defined plugin graphs written with `tf` names -----------------------------------------
@case('test_readme.py', 'ReadmeTestCase::test_custom_repr_graph')
def _custom_repr_graph():
    class Tanh(tensorrec.representation_graphs.AbstractRepresentationGraph):
        def connect_representation_graph(self, tf_features, n_components, n_features, node_name_ending):
            w = tf.Variable(tf.random_normal([n_features, n_components], stddev=.5),
                            name='tanh_weights_%s' % node_name_ending)
            return tf.nn.tanh(tf.sparse_tensor_dense_matmul(tf_features, w)), [w]

    model = tensorrec.TensorRec(user_repr_graph=Tanh(), item_repr_graph=Tanh())
    model.fit(*tensorrec.util.generate_dummy_data(num_users=100, num_items=150, interaction_density=.05), epochs=5,
              verbose=True)


@case('test_readme.py', 'ReadmeTestCase::test_custom_loss_graph')
def _custom_loss_graph():
    class MeanAbsolute(tensorrec.loss_graphs.AbstractLossGraph):
        def connect_loss_graph(self, tf_prediction_serial, tf_interactions_serial, **kwargs):
            return tf.reduce_mean(tf.abs(tf_interactions_serial - tf_prediction_serial))

    model = tensorrec.TensorRec(loss_graph=MeanAbsolute())
    model.fit(*tensorrec.util.generate_dummy_data(num_users=100, num_items=150, interaction_density=.05), epochs=5,
              verbose=True)


# ---- test_prediction_graphs.py: fit with each prediction graph; the serial forms' known answers ------------------
for _name, _graph in (('test_dot_product', PG.DotProductPredictionGraph),
                      ('test_cos_distance', PG.CosineSimilarityPredictionGraph)):
    def _fit_with_prediction(graph=_graph):
        data = generate_dummy_data_with_indicator(num_users=10, num_items=12, interaction_density=.5)
        TensorRec(prediction_graph=graph()).fit(*data, epochs=5)
    case('test_prediction_graphs.py', 'PredictionGraphsTestCase::' + _name)(_fit_with_prediction)

for _cls, _key, _graph in (('DotProductTestCase', 'dot_product_serial', PG.DotProductPredictionGraph),
                           ('CosineSimilarityTestCase', 'cosine_serial', PG.CosineSimilarityPredictionGraph),
                           ('EuclideanSimilarityTestCase', 'euclidean_serial', PG.EuclideanSimilarityPredictionGraph)):
    def _serial(key=_key, graph=_graph):
        g = GOLDEN[key]
        got = graph().connect_serial_prediction_graph(
            tf_user_representation=np.array(g['user_repr']), tf_item_representation=np.array(g['item_repr']),
            tf_x_user=np.array(g['x_user']), tf_x_item=np.array(g['x_item'])).eval(session=get_session())
        expect = np.array(g['expected']) if 'expected' in g else -np.sqrt(np.array(g['expected_neg_sqrt_of']))
        assert np.allclose(got, expect)
    case('test_prediction_graphs.py', _cls + '::test_serial_prediction')(_serial)


# ---- test_recommendation_graphs.py: known answers of the graph functions ----------------------------------------
def _rg(name):
    return case('test_recommendation_graphs.py', 'RecommendationGraphsTestCase::' + name)


@_rg('test_project_biases')
def _project_biases():
    g = GOLDEN['project_biases']
    biases, projected = project_biases(tf_features=sparse_tensor(g['features']), n_features=len(g['feature_biases']))
    get_session().run(tf.global_variables_initializer())
    get_session().run(biases.assign(value=[[b] for b in g['feature_biases']]))
    assert (projected.eval(session=get_session()) == np.array(g['expected'])).all()


@_rg('test_split_sparse_tensor_indices')
def _split():
    g = GOLDEN['split_sparse_tensor_indices']
    x_user, x_item = split_sparse_tensor_indices(tf_sparse_tensor=sparse_tensor(g['interactions']), n_dimensions=2)
    assert (x_user.eval(session=get_session()) == np.array(g['expected_user'])).all()
    assert (x_item.eval(session=get_session()) == np.array(g['expected_item'])).all()


@_rg('test_bias_prediction_serial')
def _bias_serial():
    g = GOLDEN['bias_prediction_serial']
    got = bias_prediction_serial(
        tf_prediction_serial=np.array(g['predictions'], dtype=np.float32),
        tf_projected_user_biases=np.array(g['user_biases']), tf_projected_item_biases=np.array(g['item_biases']),
        tf_x_user=np.array(g['x_user']), tf_x_item=np.array(g['x_item'])).eval(session=get_session())
    assert (got == np.array(g['expected'], dtype=np.float32)).all()


@_rg('test_densify_sampled_item_predictions')
def _densify():
    g = GOLDEN['densify_sampled_item_predictions']
    got = densify_sampled_item_predictions(tf_sample_predictions_serial=np.array(g['input']),
                                           tf_n_sampled_items=g['n_sampled_items'],
                                           tf_n_users=g['n_users']).eval(session=get_session())
    assert (got == np.array(g['expected'])).all()


def main(target):
    failed = 0
    try:
        for name, fn in CASES[target]:
            try:
                fn()
                print('PASS', name, flush=True)
            except Exception:
                failed += 1
                print('FAIL', name, flush=True)
                traceback.print_exc()
    finally:
        if _TensorRecData.ready:
            shutil.rmtree(_TensorRecData.tmp)
    return 1 if failed else 0


if __name__ == '__main__':
    sys.exit(main(sys.argv[1]))
