"""PDB pocket ingest + featurizer (SURVEY.md 8(f) n1)."""
import os

import numpy as np
import pytest
import torch

from targetdiff_b200 import atom_num
from targetdiff_b200.pocket import (AA_INDEX, featurize_protein_atoms, get_atomic_number_from_index, is_aromatic_from_index, parse_pdb_atoms,
                                    pdb_to_pocket_data)

PDB = """HEADER    POCKET
COMPND    POCKET
ATOM    219  N   LEU A  36      36.155  52.241  55.687  1.00 30.88         A N
ATOM    220  CA  LEU A  36      35.391  51.712  54.566  1.00 30.88         A C
ATOM    221  C   LEU A  36      35.560  50.200  54.537  1.00 30.88         A C
ATOM    222  O   LEU A  36      36.675  49.694  54.705  1.00 30.88         A O
ATOM    223  CB  LEU A  36      35.842  52.361  53.252  1.00 30.88         A C
ATOM    300  SG  CYS A  40      30.000  50.000  50.000  1.00 20.00
ATOM    301 SE   MSE A  41      31.000  50.000  50.000  1.00 20.00          SE
ENDMDL
ATOM    999  N   GLY A  99       0.000   0.000   0.000  1.00  0.00           N
END
"""


def test_fixed_column_parser_and_featurizer():
    with pytest.raises(KeyError):
        parse_pdb_atoms(PDB)                       # MSE is not one of the 20 residues: the reference raises KeyError as well
    block = PDB.replace('MSE', 'MET')
    d = parse_pdb_atoms(block)
    assert d['molecule_name'] == 'pocket' and len(d['element']) == 7          # the record after ENDMDL is ignored
    assert d['element'].tolist() == [7, 6, 6, 8, 6, 16, 34]                   # SG: element falls back to the atom-name column
    assert d['is_backbone'].tolist() == [True, True, True, True, False, False, False]
    assert d['atom_to_aa_type'].tolist() == [AA_INDEX['LEU']] * 5 + [AA_INDEX['CYS'], AA_INDEX['MET']]
    np.testing.assert_allclose(d['pos'][0], [36.155, 52.241, 55.687], rtol=0, atol=1e-5)
    f = featurize_protein_atoms(d['element'], d['atom_to_aa_type'], d['is_backbone'])
    assert f.shape == (7, 27) and f.dtype == torch.int64
    assert f[0, :6].tolist() == [0, 0, 1, 0, 0, 0] and f[5, :6].tolist() == [0, 0, 0, 0, 1, 0] and f[6, :6].tolist() == [0, 0, 0, 0, 0, 1]
    assert f[0, 6 + AA_INDEX['LEU']] == 1 and int(f[0, 6:26].sum()) == 1 and f[0, 26] == 1 and f[4, 26] == 0
    data = pdb_to_pocket_data(block)
    assert data.protein_pos.shape == (7, 3) and data.protein_atom_feature.shape == (7, 27) and data.ligand_pos.shape == (0, 3)


def test_ligand_class_maps():
    idx = np.arange(13)
    assert get_atomic_number_from_index(idx) == [1, 6, 6, 7, 7, 8, 8, 9, 15, 15, 16, 16, 17]
    assert is_aromatic_from_index(idx) == [False, False, True, False, True, False, True, False, False, True, False, True, False]


# the reference's examples/1h36_A_rec_1h36_r88_lig_tt_docked_0_pocket10.pdb, byte for byte
PDB_1H36 = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', '1h36_pocket10.pdb')


def test_1h36_pocket_matches_survey_facts():
    data = pdb_to_pocket_data(PDB_1H36)
    el = data.protein_element.tolist()
    assert len(el) == 572 and (el.count(6), el.count(7), el.count(8), el.count(16)) == (374, 87, 109, 2)      # SURVEY.md 8(c)
    assert len(set(data.protein_atom_to_aa_type.tolist())) == 19
    assert atom_num.get_space_size(data.protein_pos.numpy()) == pytest.approx(38.37, abs=0.01)
    assert atom_num._get_bin_idx(atom_num.get_space_size(data.protein_pos.numpy())) == 9
    assert data.protein_atom_feature.sum(-1).min() >= 2
