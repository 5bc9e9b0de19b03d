"""Shared helpers of the Tacotron tests: weights (shipped checkpoint or portable synthetic), sentences."""
import json
import os

import numpy as np

from conftest import GOLDEN, ROOT

TRAVEL_COPY = os.path.join(ROOT, 'oracle', '_ref', 'tacotron_weights.npz')

SHAPES = {
    'inputs_embedding': (191, 128),
    'memory_layer/kernel': (512, 128),
    'decoder/Location_Sensitive_Attention/query_layer/kernel': (256, 128),
    'decoder/Location_Sensitive_Attention/location_features_convolution/kernel': (31, 1, 32),
    'decoder/Location_Sensitive_Attention/location_features_convolution/bias': (32,),
    'decoder/Location_Sensitive_Attention/location_features_layer/kernel': (32, 128),
    'decoder/Location_Sensitive_Attention/attention_variable_projection': (128,),
    'decoder/Location_Sensitive_Attention/attention_bias': (128,),
    'decoder/decoder_prenet/dense_1/kernel': (80, 256), 'decoder/decoder_prenet/dense_1/bias': (256,),
    'decoder/decoder_prenet/dense_2/kernel': (256, 256), 'decoder/decoder_prenet/dense_2/bias': (256,),
    'decoder/decoder_LSTM/multi_rnn_cell/cell_0/decoder_LSTM_1/kernel': (1024, 1024),
    'decoder/decoder_LSTM/multi_rnn_cell/cell_0/decoder_LSTM_1/bias': (1024,),
    'decoder/decoder_LSTM/multi_rnn_cell/cell_1/decoder_LSTM_2/kernel': (512, 1024),
    'decoder/decoder_LSTM/multi_rnn_cell/cell_1/decoder_LSTM_2/bias': (1024,),
    'decoder/dense/kernel': (768, 1), 'decoder/dense/bias': (1,),
    'decoder/linear_transform_projection/projection_linear_transform_projection/kernel': (768, 80),
    'decoder/linear_transform_projection/projection_linear_transform_projection/bias': (80,),
    'decoder/stop_token_projection/projection_stop_token_projection/kernel': (768, 1),
    'decoder/stop_token_projection/projection_stop_token_projection/bias': (1,),
}


def synth_taco_weights(seed=0):
    """Portable random weights with the checkpoint's decoder shapes (numpy legacy RNG)."""
    rs = np.random.RandomState(seed)
    w = {}
    for k, shp in SHAPES.items():
        fan_in = shp[0] if len(shp) > 1 else 16
        scale = 1.0 / np.sqrt(fan_in)
        if k.endswith('decoder_LSTM_1/kernel') or k.endswith('decoder_LSTM_2/kernel'):
            scale *= 2.0
        w[k] = rs.uniform(-scale, scale, size=shp).astype(np.float32) * (1.0 if len(shp) > 1 else 0.3)
    return w


def real_taco_weights():
    """The shipped checkpoint's inference variables, from the copy __graft_entry__.build() makes under oracle/_ref/, or None."""
    if os.path.isfile(TRAVEL_COPY):
        return dict(np.load(TRAVEL_COPY))
    return None


def sentences():
    return json.load(open(os.path.join(GOLDEN, 'taco_symbols.json')))
