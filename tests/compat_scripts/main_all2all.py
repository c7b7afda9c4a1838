"""Every node merges all its neighbours' models with mixing weights, written against the original gossipy API
(``from gossipy ...``).  tests/test_compat.py runs it unmodified through ``python -m gossipy_b200.compat``."""
import networkx as nx
import torch

from gossipy import set_seed
from gossipy.core import AntiEntropyProtocol, CreateModelMode, StaticP2PNetwork, UniformMixing
from gossipy.data import DataDispatcher, load_classification_dataset
from gossipy.data.handler import ClassificationDataHandler
from gossipy.model.handler import WeightedTMH
from gossipy.model.nn import LogisticRegression
from gossipy.node import All2AllGossipNode
from gossipy.simul import All2AllGossipSimulator, SimulationReport
from gossipy.utils import plot_evaluation

N_NODES = 40

set_seed(31)
X, y = load_classification_dataset("breast", as_tensor=True)          # bundled with scikit-learn: no download
handler = ClassificationDataHandler(X, y, test_size=.2)
dispatcher = DataDispatcher(handler, n=N_NODES, eval_on_user=False, auto_assign=True)
topology = StaticP2PNetwork(N_NODES, topology=nx.to_numpy_array(nx.random_regular_graph(4, N_NODES, seed=3)))
proto = WeightedTMH(net=LogisticRegression(handler.Xtr.shape[1], 2), optimizer=torch.optim.SGD,
                    optimizer_params={"lr": .2, "weight_decay": .001}, criterion=torch.nn.CrossEntropyLoss(),
                    create_model_mode=CreateModelMode.MERGE_UPDATE)
nodes = All2AllGossipNode.generate(data_dispatcher=dispatcher, p2p_net=topology, model_proto=proto, round_len=30, sync=False)

simulator = All2AllGossipSimulator(nodes=nodes, data_dispatcher=dispatcher, delta=30, protocol=AntiEntropyProtocol.PUSH,
                                   sampling_eval=.2)
report = SimulationReport()
simulator.add_receiver(report)
simulator.init_nodes(seed=9)
simulator.start(UniformMixing(topology), n_rounds=100)
plot_evaluation([[ev for _, ev in report.get_evaluation(local=False)]], "Global test set")
