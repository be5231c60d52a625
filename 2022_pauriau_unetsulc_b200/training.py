"""``UnetTrainingSulciLabelling`` — full training of the UNet3D on a cohort (reference training.py:33-299).

Keeps the reference's public surface (constructor, ``load_network``, ``learning``, ``reset_results``, result keys,
tensorboard layout ``<working_path>/tensorboard/<model>/cv<k>``) and its semantics: SGD(lr, momentum, wd 0) +
CrossEntropyLoss(ignore_index=-1), train then val phase per epoch, val loss on the eval-mode (softmax) outputs,
best weights by strict ``val acc >``, DivideLr(patience, repeat=1) dividing lr by 10 and resetting momentum,
EarlyStopping on the val loss.
"""
import os

from .early_stopping import DivideLr
from .models import UNet3D
from .pattern_class import UnetPatternSulciLabelling, make_head

_RESULT_KEYS = ('lr', 'momentum', 'batch_size', 'num_epochs', 'graphs_train', 'graphs_test', 'epoch_loss_val',
                'epoch_acc_val', 'epoch_loss_train', 'epoch_acc_train', 'best_acc', 'best_epoch', 'divide_lr_epoch',
                'duration')


def _empty_results(extra=()):
    res = {k: [] for k in _RESULT_KEYS + tuple(extra)}
    res['patience'] = {}
    res['threshold_scores'] = {}
    return res


class UnetTrainingSulciLabelling(UnetPatternSulciLabelling):

    def __init__(self, graphs, hemi, cuda=-1, working_path=None, dict_model={},
                 dict_names=None, dict_bck2=None, sulci_side_list=None):
        super().__init__(graphs, hemi, cuda, working_path, dict_model, dict_names, dict_bck2, sulci_side_list)
        self.results = _empty_results()

    def load_network(self):
        print('Network initialization...')
        self.model = UNet3D(self.num_channel, len(self.sulci_side_list), final_sigmoid=self.final_sigmoid,
                            interpolate=self.interpolate, dropout=0., conv_layer_order=self.conv_layer_order,
                            init_channel_number=self.num_filter, conv_bias=self.conv_bias)
        if self.num_conv > 1:
            # the reference reads an undefined self.dict_trained_model here (training.py:69); the filter count of
            # this model is the intended value
            self.model.final_conv = make_head(self.num_filter, len(self.sulci_side_list), self.num_conv)
        self.model = self.model.to(self.device)

    def learning(self, lr, momentum, num_epochs, gfile_list_train, gfile_list_test, batch_size=1, patience={},
                 save_results=True):
        if self.sulci_side_list is None or self.dict_bck2 is None or self.dict_names is None:
            print('Error : extract data from graphs before learning')
            return 1
        trainloader, valloader, sizes = self._loaders(gfile_list_train, gfile_list_test, batch_size, num_epochs)
        self.load_network()

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
                tr, va = [int(i) for i in sizes['train']], [int(i) for i in sizes['val']]
                if num_training == 0:
                    self.results['train_image_size'], self.results['val_image_size'] = tr, va
                else:
                    self.results['train_image_size'].append(tr)
                    self.results['val_image_size'].append(va)
        tb_dir = os.path.join(self.working_path + '/tensorboard/' + self.model_name, 'cv' + str(num_training))
        if save_results:
            os.makedirs(os.path.dirname(tb_dir), exist_ok=True)

        divide_lr = DivideLr(patience=patience['divide_lr']) if 'divide_lr' in patience else None

        def after_epoch(epoch, val_loss, state):
            if divide_lr is None:
                return
            divide_lr(val_loss, self.model)
            if divide_lr.divide_lr:
                state['lr'] = state['lr'] / 10
                state['new_optimizer'] = True
                print('\tDivide learning rate. New value: {}'.format(state['lr']))
                self.results['divide_lr_epoch'].append(epoch)

        self._fit(lr, momentum, num_epochs, trainloader, valloader, patience, save_results, num_training, tb_dir,
                  after_epoch=after_epoch)

    def reset_results(self):
        self.results = _empty_results(extra=('train_image_size', 'val_image_size'))
