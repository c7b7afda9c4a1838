"""Pegasos with one training sample per node, written against the original gossipy API (``from gossipy ...``).

tests/test_compat.py runs it unmodified through ``python -m gossipy_b200.compat --engine native``: 1 617 nodes of a
linear learner on a clique with churn, message loss and delays, the set-up the banked engine takes over."""
from gossipy import set_seed
from gossipy.core import AntiEntropyProtocol, CreateModelMode, StaticP2PNetwork, UniformDelay
from gossipy.data import DataDispatcher, load_classification_dataset
from gossipy.data.handler import ClassificationDataHandler
from gossipy.model.handler import PegasosHandler
from gossipy.model.nn import AdaLine
from gossipy.node import GossipNode
from gossipy.simul import GossipSimulator, SimulationReport
from gossipy.utils import plot_evaluation

set_seed(11)
X, y = load_classification_dataset("digits", as_tensor=True)          # bundled with scikit-learn: no download
y = 2 * (y >= 5).long() - 1                                           # digits 0-4 against 5-9, labels -1 / +1
handler = ClassificationDataHandler(X, y, test_size=.1)
dispatcher = DataDispatcher(handler, eval_on_user=False, auto_assign=True)   # no n: one training sample per node
proto = PegasosHandler(net=AdaLine(handler.size(1)), learning_rate=.02, create_model_mode=CreateModelMode.MERGE_UPDATE)
nodes = GossipNode.generate(data_dispatcher=dispatcher, p2p_net=StaticP2PNetwork(dispatcher.size(), None),
                            model_proto=proto, round_len=20, sync=False)

simulator = GossipSimulator(nodes=nodes, data_dispatcher=dispatcher, delta=20, protocol=AntiEntropyProtocol.PUSH,
                            delay=UniformDelay(0, 4), online_prob=.5, drop_prob=.05, sampling_eval=.05)
report = SimulationReport()
simulator.add_receiver(report)
simulator.init_nodes(seed=5)
simulator.start(n_rounds=50)
plot_evaluation([[ev for _, ev in report.get_evaluation(False)]], "Global test set")
