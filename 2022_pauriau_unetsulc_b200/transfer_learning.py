"""``UnetTransferSulciLabelling`` — transfer learning from a trained ``.mdsm`` (reference
transfer_learning/transfer_learning.py:27-416), in the new-style layout the reference's top-level main.py expects
(``from transfer_learning import UnetTransferSulciLabelling``; inherits the base class; no positional
``translation_file`` — passing one as a keyword is still accepted).

Semantics kept: the trained UNet3D is rebuilt with ITS number of outputs, loaded, deep-copied and given a fresh
``final_conv`` (seed 42); every train step sets ``requires_grad`` by name prefix from ``training_layers``
(default ``['final_conv']``) so frozen layers get no gradient and are skipped by SGD; after ``patience['fine_tunning']``
non-improving val losses, or at epoch ``int(0.8*num_epochs)``, ``fine_tunning_layers`` (default decoders.2/1/0) are
added IN PLACE to ``training_layers`` (it aliases ``dict_model['training_layers']`` and persists across CV folds, as
in the reference), lr is divided by 10 and the optimiser rebuilt.
On the B200 path freezing prunes work: phase A runs no dgrad/wgrad at all below the head; phase B stops the
backward pass at ``decoders.0`` (no gradient ever enters the encoders).
"""
import copy
import os

import torch

from .early_stopping import FineTunning
from .models import UNet3D
from .pattern_class import UnetPatternSulciLabelling, make_head
from .training import _empty_results


class UnetTransferSulciLabelling(UnetPatternSulciLabelling):

    def __init__(self, graphs, hemi, cuda=-1, working_path=None, dict_model={}, dict_trained_model={},
                 dict_names=None, dict_bck2=None, sulci_side_list=None, translation_file=None):
        super().__init__(graphs, hemi, cuda, working_path, dict_model, dict_names, dict_bck2, sulci_side_list)
        self.training_layers = dict_model.get('training_layers', ['final_conv'])
        self.fine_tunning_layers = dict_model.get('fine_tunning_layers', ['decoders.2', 'decoders.1', 'decoders.0'])
        self.dict_trained_model = dict_trained_model
        self.results = self._fresh_results()
        if translation_file is not None and os.path.exists(translation_file):
            import sigraph
            self.flt = sigraph.FoldLabelsTranslator()
            self.flt.readLabels(translation_file)
            self.trfile = translation_file

    @staticmethod
    def _fresh_results():
        res = _empty_results(extra=('fine_tunning_epoch',))
        res.pop('divide_lr_epoch')
        return res

    def reset_results(self):
        self.results = self._fresh_results()

    def load_model(self):
        print('Network initialization...')
        tm = self.dict_trained_model = self.fill_dict_model(self.dict_trained_model)
        torch.manual_seed(42)
        print('Model_file: ', tm['model_file'])
        trained = UNet3D(tm['in_channels'], tm['out_channels'], final_sigmoid=tm['final_sigmoid'],
                         interpolate=tm['interpolate'], conv_layer_order=tm['conv_layer_order'],
                         init_channel_number=tm['init_channel_number'], conv_bias=tm.get('conv_bias', False))
        if tm.get('num_conv', 1) > 1:
            trained.final_conv = make_head(tm['init_channel_number'], tm['out_channels'], tm['num_conv'])
        trained.load_state_dict(torch.load(tm['model_file'], map_location='cpu'))
        self.model = copy.deepcopy(trained)
        self.model.final_conv = make_head(tm['init_channel_number'], len(self.sulci_side_list), self.num_conv)
        self.model = self.model.to(self.device)

    def _apply_freeze_mask(self):
        for name, p in self.model.named_parameters():
            p.requires_grad = any(name.startswith(layer) for layer in self.training_layers)

    def learning(self, lr, momentum, num_epochs, gfile_list_train, gfile_list_test, batch_size=1, patience={},
                 save_results=True):
        if self.sulci_side_list is None or self.dict_bck2 is None or self.dict_names is None:
            print('Error : extract data from graphs before learning')
            return 1
        trainloader, valloader, sizes = self._loaders(gfile_list_train, gfile_list_test, batch_size, num_epochs)
        self.load_model()

        num_training = len(self.results['lr'])
        if save_results:
            self.results['lr'].append(lr)
            self.results['momentum'].append(momentum)
            self.results['batch_size'].append(batch_size)
            self.results['num_epochs'].append(num_epochs)
            self.results['graphs_test'].append(list(gfile_list_test))
            self.results['graphs_train'].append(list(gfile_list_train))
            self.results['patience'] = patience
            if batch_size > 1:
                self.results.setdefault('train_image_size', []).append([int(i) for i in sizes['train']])
                self.results.setdefault('val_image_size', []).append([int(i) for i in sizes['val']])
        tb_dir = os.path.join(self.working_path + '/tensorboard/' + self.model_name, 'cv_' + str(num_training))
        if save_results:
            os.makedirs(os.path.dirname(tb_dir), exist_ok=True)

        fine_tunning = FineTunning(patience=patience['fine_tunning'], save=False) if 'fine_tunning' in patience else None

        def after_epoch(epoch, val_loss, state):
            if fine_tunning is None:
                return
            fine_tunning(val_loss, self.model)
            if epoch == int(0.8 * num_epochs):
                fine_tunning.ft_start = True
                fine_tunning.stop = True
            if fine_tunning.ft_start:
                print('\nFine tunning')
                self.training_layers += self.fine_tunning_layers      # in place, on purpose (see module docstring)
                state['lr'] = state['lr'] / 10
                state['new_optimizer'] = True
                print('Divide learning rate. New value: {}\n'.format(state['lr']))
                if save_results:
                    self.results['fine_tunning_epoch'].append(epoch)

        self._fit(lr, momentum, num_epochs, trainloader, valloader, patience, save_results, num_training, tb_dir,
                  before_step=self._apply_freeze_mask, after_epoch=after_epoch)
