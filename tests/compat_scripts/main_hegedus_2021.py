"""Partitioned models under token-account flow control, written against the original gossipy API (``from gossipy ...``).

tests/test_compat.py runs it unmodified through ``python -m gossipy_b200.compat``, on the Python loop and on the C++
scheduler + executor: a tokenized simulation of PartitioningBasedNode / PartitionedTMH with a constant utility."""
import torch
from networkx import to_numpy_array
from networkx.generators.random_graphs import random_regular_graph

from gossipy import set_seed
from gossipy.core import AntiEntropyProtocol, CreateModelMode, StaticP2PNetwork, UniformDelay
from gossipy.data import DataDispatcher, load_classification_dataset
from gossipy.data.handler import ClassificationDataHandler
from gossipy.flow_control import RandomizedTokenAccount
from gossipy.model.handler import PartitionedTMH
from gossipy.model.nn import LogisticRegression
from gossipy.model.sampling import TorchModelPartition
from gossipy.node import PartitioningBasedNode
from gossipy.simul import SimulationReport, TokenizedGossipSimulator
from gossipy.utils import plot_evaluation

N_NODES = 50

set_seed(2024)
X, y = load_classification_dataset("breast", as_tensor=True)          # bundled with scikit-learn: no download
handler = ClassificationDataHandler(X, y, test_size=.2)
dispatcher = DataDispatcher(handler, n=N_NODES, eval_on_user=False, auto_assign=True)
graph = StaticP2PNetwork(N_NODES, to_numpy_array(random_regular_graph(6, N_NODES, seed=7)))
net = LogisticRegression(handler.Xtr.shape[1], 2)
proto = PartitionedTMH(net=net, tm_partition=TorchModelPartition(net, 3), optimizer=torch.optim.SGD,
                       optimizer_params={"lr": .5, "weight_decay": .01}, criterion=torch.nn.CrossEntropyLoss(),
                       create_model_mode=CreateModelMode.UPDATE)
nodes = PartitioningBasedNode.generate(data_dispatcher=dispatcher, p2p_net=graph, model_proto=proto, round_len=50, sync=True)

simulator = TokenizedGossipSimulator(nodes=nodes, data_dispatcher=dispatcher, token_account=RandomizedTokenAccount(C=3, A=1),
                                     utility_fun=lambda mh1, mh2, msg: 1, delta=50, protocol=AntiEntropyProtocol.PUSH,
                                     delay=UniformDelay(0, 5), sampling_eval=.2)
report = SimulationReport()
simulator.add_receiver(report)
simulator.init_nodes(seed=3)
simulator.start(n_rounds=200)
plot_evaluation([[ev for _, ev in report.get_evaluation(False)]], "Global test set")
