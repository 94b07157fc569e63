# Written for tests/test_host_logic.py in the format of the reference's tensorflowdata/*/conf.py (SURVEY.md section 5):
# multi-object flow model with a missing comma after 'learning_rate' -- the reference's own file of this name does not parse.
import os
current_dir = os.path.dirname(os.path.realpath(__file__))
from multiobject_appflow import MultiObjectAppFlow

configuration = {
    'experiment_name': os.path.basename(current_dir),
    'data_dir': current_dir + '/data',
    'output_dir': current_dir + '/modeldata',
    'current_dir': current_dir,
    'num_iterations': 200000,
    'batch_size': 64,
    'learning_rate': 1e-4
    'train_val_split': 0.95,
    'use_color': '',
    'use_depth': 0.1,
    'model': MultiObjectAppFlow,
}
