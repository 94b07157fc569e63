# Written for tests/test_host_logic.py in the format of the reference's tensorflowdata/*/conf.py (SURVEY.md section 5):
# no 'model' key: train.py falls back to Base_Prediction_Model; colour and depth heads are key-presence switches.
import os
current_dir = os.path.dirname(os.path.realpath(__file__))

configuration = {
    'experiment_name': os.path.basename(current_dir),
    'data_dir': current_dir + '/data',
    'output_dir': current_dir + '/modeldata',
    'current_dir': current_dir,
    'num_iterations': 200000,
    'batch_size': 64,
    'learning_rate': 1e-4,
    'train_val_split': 0.95,
    'use_color': '',
    'use_depth': '',
    'depth_lr_factor': 0.1,
}
