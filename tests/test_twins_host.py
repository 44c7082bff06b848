"""Which forward activations of a 16-bit grad plan get a bf16 twin: those a dense (GEMM) weight gradient reads, and no
other (the grouped-conv weight gradient reads the fp16 activation itself).  Host logic only."""
from nb_asr_b200.engine import dense_wgrad_inputs
from nb_asr_b200.model import CELLS_PER_BLOCK
from nb_asr_b200.search_space import arch_vec_to_names

DEFAULT = [[1, 0], [1, 0, 0], [1, 0, 0, 0]]          # conv5 x 3, no skips
LINEAR_SKIPS = [[0, 1], [0, 1, 1], [0, 1, 1, 1]]
MIXED = [[2, 1], [3, 0, 1], [0, 1, 0, 1]]            # conv5d2, conv7, linear


def block_outputs(use_norm, last_node=2):
    """name of the last cell output of blocks 0..2: the next block's time-reduction conv input"""
    return {(f'b{i}.c{CELLS_PER_BLOCK[i] - 1}.ln' if use_norm else f'b{i}.c{CELLS_PER_BLOCK[i] - 1}.n{last_node}') for i in range(3)}


def test_default_arch_keeps_only_block_inputs_and_lstm_input():
    got = dense_wgrad_inputs(arch_vec_to_names(DEFAULT), True, True)
    assert got == {'input', 'b3.c5.ln'} | block_outputs(True)
    assert dense_wgrad_inputs(arch_vec_to_names(DEFAULT), True, True, input_dropout=True) == {'input', 'lstm_in'} | block_outputs(True)


def test_without_rnn_the_encoder_output_has_no_twin():
    assert dense_wgrad_inputs(arch_vec_to_names(DEFAULT), True, False) == {'input'} | block_outputs(True)
    assert dense_wgrad_inputs(arch_vec_to_names(DEFAULT), True, False, input_dropout=True) == {'input'} | block_outputs(True)


def test_without_norm_cell_outputs_are_last_node_outputs():
    got = dense_wgrad_inputs(arch_vec_to_names(DEFAULT), False, True)
    assert got == {'input', 'b3.c5.n2'} | block_outputs(False)


def test_linear_edges_read_twins_of_their_inputs():
    ln = arch_vec_to_names(LINEAR_SKIPS)
    got = dense_wgrad_inputs(ln, True, True)
    want = {'input', 'b3.c5.ln'} | block_outputs(True)
    for i, nc in enumerate(CELLS_PER_BLOCK):
        for c in range(nc):
            # node 0 reads the cell input (block LayerNorm for cell 0, else the previous cell's LayerNorm), node n > 0 reads
            # node n-1's output
            want |= {f'b{i}.ln' if c == 0 else f'b{i}.c{c - 1}.ln', f'b{i}.c{c}.n0', f'b{i}.c{c}.n1'}
    assert got == want
    # without norm the cell input of cell c > 0 is the previous cell's last node output
    got = dense_wgrad_inputs(ln, False, False)
    want = {'input'} | block_outputs(False)
    for i, nc in enumerate(CELLS_PER_BLOCK):
        for c in range(nc):
            want |= {f'b{i}.ln' if c == 0 else f'b{i}.c{c - 1}.n2', f'b{i}.c{c}.n0', f'b{i}.c{c}.n1'}
    assert got == want


def test_mixed_arch_twins_only_the_linear_node_input():
    got = dense_wgrad_inputs(arch_vec_to_names(MIXED), True, True)
    want = {'input', 'b3.c5.ln'} | block_outputs(True)
    for i, nc in enumerate(CELLS_PER_BLOCK):
        want |= {f'b{i}.c{c}.n1' for c in range(nc)}       # node 2 (linear) reads node 1's output
    assert got == want
